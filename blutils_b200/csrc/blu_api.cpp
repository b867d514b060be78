// blu_api.cpp -- C ABI (include/blu_consensus.h): context, taxonomy upload, chunked streaming of the outfmt-6
// text through the CUDA kernels, result download/decoding and the reference-compatible writer.
//
// There is deliberately NO CPU implementation of the consensus here: everything that computes goes through
// blu_kernels.cu; without a CUDA device every compute entry point fails with BLU_ERR_CUDA.
#include <cuda_runtime.h>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cerrno>
#include <cstdio>
#include <cstring>
#include <exception>
#include <filesystem>
#include <fstream>
#include <memory>
#include <mutex>
#include <random>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/blu_consensus.h"
#include "blu_decode.h"
#include "blu_json.h"
#include "blu_kernels.h"
#include "blu_sort.h"
#include "blu_tabular.h"
#include "blu_taxonomy.h"

using namespace blu;

namespace {

thread_local std::string g_create_error;

struct CudaErr : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct UnsupportedErr : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define CK(expr)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) throw CudaErr(std::string(#expr) + ": " + cudaGetErrorString(_e));       \
    } while (0)

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        CK(cudaMalloc((void**)&p, n * sizeof(T)));
        cap = n;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// One cudaMalloc'ed block freed by its owner: an uploaded or regrouped table, a sort's scratch.
struct DevMem {
    uint8_t* p = nullptr;
    uint64_t n = 0;  // bytes of text it holds
    DevMem() = default;
    DevMem(const DevMem&) = delete;
    DevMem& operator=(const DevMem&) = delete;
    ~DevMem() {
        if (p) cudaFree(p);
    }
    bool alloc(uint64_t bytes) {  // false: the device is full (the error is cleared)
        if (cudaMalloc((void**)&p, std::max<uint64_t>(bytes, 1)) == cudaSuccess) return true;
        cudaGetLastError();
        p = nullptr;
        return false;
    }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// Pinned result buffers are recycled between runs.  The pool is shared by the context and every result it
// produced, so a result may be freed after its context.
struct PinnedPool {
    std::mutex mu;
    std::vector<PinnedBuf> free_list;
    bool closed = false;
    PinnedBuf acquire(size_t bytes) {
        {
            std::lock_guard<std::mutex> g(mu);
            size_t best = SIZE_MAX;
            for (size_t i = 0; i < free_list.size(); i++)
                if (free_list[i].cap >= bytes && (best == SIZE_MAX || free_list[i].cap < free_list[best].cap)) best = i;
            if (best != SIZE_MAX) {
                PinnedBuf b = free_list[best];
                free_list.erase(free_list.begin() + best);
                return b;
            }
        }
        PinnedBuf b;
        size_t cap = std::max<size_t>(bytes + bytes / 8, 4096);
        CK(cudaHostAlloc(&b.p, cap, cudaHostAllocDefault));
        b.cap = cap;
        return b;
    }
    void release(PinnedBuf b) {
        if (!b.p) return;
        {
            std::lock_guard<std::mutex> g(mu);
            if (!closed && free_list.size() < 16) {
                free_list.push_back(b);
                return;
            }
        }
        cudaFreeHost(b.p);
    }
    void close() {
        std::vector<PinnedBuf> v;
        {
            std::lock_guard<std::mutex> g(mu);
            closed = true;
            v.swap(free_list);
        }
        for (auto& b : v) cudaFreeHost(b.p);
    }
};

}  // namespace

namespace {

// Result arrays on the device (records / beans / accession references).  A device-resident result takes the set it
// was computed into with it and hands it back when it is freed, so back-to-back runs never wait for cudaMalloc.
struct DeviceSet {
    DevBuf<blu_record> rec;
    DevBuf<blu_bean> beans;
    DevBuf<blu_acc> accs;
    void release() { rec.release(), beans.release(), accs.release(); }
};

struct DevicePool {
    std::mutex mu;
    std::vector<std::unique_ptr<DeviceSet>> free_list;
    int device = 0;
    bool closed = false;
    std::unique_ptr<DeviceSet> acquire() {
        std::lock_guard<std::mutex> g(mu);
        if (free_list.empty()) return std::make_unique<DeviceSet>();
        // the largest set: fewest reallocations
        size_t best = 0;
        for (size_t i = 1; i < free_list.size(); i++)
            if (free_list[i]->rec.cap > free_list[best]->rec.cap) best = i;
        auto s = std::move(free_list[best]);
        free_list.erase(free_list.begin() + best);
        return s;
    }
    void release(std::unique_ptr<DeviceSet> s) {
        if (!s) return;
        {
            std::lock_guard<std::mutex> g(mu);
            if (!closed && free_list.size() < 4) {
                free_list.push_back(std::move(s));
                return;
            }
        }
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(device);
        s->release();
        cudaSetDevice(cur);
    }
    void close() {
        std::vector<std::unique_ptr<DeviceSet>> v;
        {
            std::lock_guard<std::mutex> g(mu);
            closed = true;
            v.swap(free_list);
        }
        for (auto& s : v) s->release();
    }
};

constexpr int kMaxRanges = 8;  // ranges of a resident table / event sets kept per context

}  // namespace

struct blu_ctx {
    blu_opts opts{};
    Cutoffs cut;
    int device = 0;
    int sms = 148;
    cudaStream_t stream = nullptr, copy_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev[kMaxRanges][4]{};  // per range / chunk: before tile, after tile, after long-run, after the post-pass
    cudaEvent_t ev_h2d[2]{}, ev_free[2]{};
    std::shared_ptr<HostTaxonomy> tax;
    // device taxonomy
    DevBuf<uint32_t> d_lin_off, d_lvl, d_bean, d_irank;
    DevBuf<double> d_cut;
    DevBuf<uint16_t> d_rcls, d_acls;
    DevBuf<uint8_t> d_linok;
    DevBuf<HashSlot> d_slots;
    LinTables dT{};
    // run buffers
    DevBuf<uint8_t> d_text[2];
    std::unique_ptr<DeviceSet> out;  // records / beans / accession references of the run in progress
    DevBuf<TopRowRaw> d_top;
    DevBuf<uint64_t> d_defer;
    DevBuf<uint8_t> d_pool;
    DevBuf<unsigned long long> d_dup, d_qhash;
    DevBuf<TopRow> d_big_rows;
    DevBuf<unsigned long long> d_big_cand;
    Counters* d_ctr = nullptr;
    Counters* h_snap = nullptr;  // pinned + mapped: kMaxRanges snapshots written by advance_kernel
    Counters* d_snap = nullptr;  // device alias of h_snap
    std::shared_ptr<PinnedPool> pool = std::make_shared<PinnedPool>();
    std::shared_ptr<DevicePool> dev_pool = std::make_shared<DevicePool>();
    std::string err;
    blu_timings tm{};
    uint64_t carry_bytes = 64ull << 20;
    // output densities (per text byte) learnt from earlier runs / the probe: capacities are sized from them
    double dens_rec = 0, dens_slot = 0, dens_bean = 0, dens_acc = 0, dens_pool = 0;
    // a multi-device context owns one single-device context per GPU and nothing else
    std::vector<std::unique_ptr<blu_ctx>> shards;
    bool keep_hashes = false;  // a shard of a multi-device context keeps every record's id hash for the cross-shard duplicate check
    bool is_multi() const { return !shards.empty(); }

    PinnedBuf acquire(size_t bytes) { return pool->acquire(bytes); }
};

// One part of a result: what one GPU produced.
struct ResultPartOwned {
    std::shared_ptr<PinnedPool> pinned;
    PinnedBuf b_rec, b_beans, b_accs, b_pool;
    const char* ext_strings = nullptr;  // BLU_OPT_TEXT_REFS: the caller's text the string references point into
    uint64_t ext_len = 0;
    uint64_t n_rec = 0, n_beans = 0, n_accs = 0, pool_len = 0;
    // device-resident results
    std::shared_ptr<DevicePool> dev_pool;
    std::unique_ptr<DeviceSet> dev;
    blu_ctx* ctx = nullptr;            // (download needs the context's streams and kernels)
    const uint8_t* dtext = nullptr;    // the device text the references point into
    std::shared_ptr<uint8_t> owned_dtext;  // ... when it is the library's regrouped copy of a scattered table (freed with the result)
    uint64_t dtext_len = 0;
    bool on_host = true;
    const char* strings() const { return ext_strings ? ext_strings : (const char*)b_pool.p; }
    uint64_t strings_len() const { return ext_strings ? ext_len : pool_len; }
    void free_buffers() {
        if (pinned) {
            pinned->release(b_rec), pinned->release(b_beans), pinned->release(b_accs), pinned->release(b_pool);
            b_rec = b_beans = b_accs = b_pool = PinnedBuf{};
        }
        if (dev_pool && dev) dev_pool->release(std::move(dev));
    }
};

struct blu_result {
    std::shared_ptr<HostTaxonomy> tax;
    Cutoffs cut;
    std::vector<ResultPartOwned> parts;
    uint64_t n_rows = 0;
    std::vector<std::string> hitless;  // NoConsensusFound (mod.rs:84-102)
    bool sorted = false;               // the records are in query-id order (blu_result_sort_by_query)
    // concatenation of a multi-part result for the array accessors (built on first use)
    mutable std::mutex merge_mu;
    mutable bool merged = false;
    mutable std::vector<blu_record> m_rec;
    mutable std::vector<blu_bean> m_beans;
    mutable std::vector<blu_acc> m_accs;
    mutable std::string m_pool;
    mutable const char* m_ext = nullptr;  // all parts reference the caller's text: the concatenation's string base is that text
    mutable uint64_t m_ext_len = 0;
    uint64_t n_rec() const {
        uint64_t n = 0;
        for (auto& p : parts) n += p.n_rec;
        return n;
    }
    bool on_host() const {
        for (auto& p : parts)
            if (!p.on_host) return false;
        return true;
    }
};

namespace {

ResultView make_view(const blu_result* r) {
    ResultView v;
    v.tax = r->tax.get();
    v.cut = r->cut;
    for (auto& p : r->parts) {
        ResultPart q;
        q.rec = (const blu_record*)p.b_rec.p;
        q.beans = (const blu_bean*)p.b_beans.p;
        q.accs = (const blu_acc*)p.b_accs.p;
        q.pool = p.strings();
        q.n_rec = p.on_host ? p.n_rec : 0;
        v.parts.push_back(q);
    }
    v.hitless_ = &r->hitless;
    v.sorted = r->sorted;
    return v;
}

int fail(blu_ctx* ctx, int code, const std::string& msg) {
    if (ctx)
        ctx->err = msg;
    else
        g_create_error = msg;
    return code;
}

template <class F>
int guarded(blu_ctx* ctx, F&& f) {
    try {
        f();
        if (ctx) ctx->err.clear();
        return BLU_OK;
    } catch (const IoErr& e) {
        return fail(ctx, BLU_ERR_IO, e.what());
    } catch (const DataErr& e) {
        return fail(ctx, BLU_ERR_DATA, e.what());
    } catch (const CudaErr& e) {
        return fail(ctx, BLU_ERR_CUDA, e.what());
    } catch (const UnsupportedErr& e) {
        return fail(ctx, BLU_ERR_UNSUPPORTED, e.what());
    } catch (const std::invalid_argument& e) {
        return fail(ctx, BLU_ERR_UNSUPPORTED, e.what());
    } catch (const std::bad_alloc&) {
        return fail(ctx, BLU_ERR_INTERNAL, "out of host memory");
    } catch (const std::exception& e) {
        return fail(ctx, BLU_ERR_INTERNAL, e.what());
    }
}

const char* dev_err_text(uint32_t e) {
    switch (e) {
        case DE_BAD_FIELD_COUNT: return "row does not have 13 tab-separated fields";
        case DE_BAD_NUMBER: return "malformed numeric field";
        case DE_EMPTY_STRING: return "empty qseqid / saccver";
        case DE_QUOTE_OR_CR: return "'\"' or '\\r' byte in the blast output (not supported)";
        case DE_UNMAPPED_TAXID: return "subject taxid of a top bit-score hit has no lineage in the taxonomy file (reference: panic on `null` lineage)";
        case DE_BAD_LINEAGE: return "Unexpected error on parse taxonomy (lineage of a top bit-score hit)";
        case DE_EMPTY_ADJUSTED: return "No taxonomy found for result (single match below every identity cutoff)";
        case DE_ROOT_DISAGREE: return "top hits disagree at the first lineage level (reference: index underflow panic)";
        case DE_BITS_RANGE: return "bit score outside the i64 range";
        case DE_NUM_UNSUPPORTED: return "number outside the exactly-parsed range (more than 19 significant digits or |exponent| > 22)";
        case DE_TOPGROUP_TOO_BIG: return "top bit-score group larger than 8192 rows";
        case DE_CARRY_TOO_BIG: return "a single row does not fit the 60 KB window";
        default: return "internal device error";
    }
}

void upload_taxonomy(blu_ctx* c) {
    HostTaxonomy& T = *c->tax;
    auto up = [&](auto& dbuf, const auto& vec) {
        dbuf.ensure(std::max<size_t>(vec.size(), 1));
        if (!vec.empty()) CK(cudaMemcpy(dbuf.p, vec.data(), vec.size() * sizeof(vec[0]), cudaMemcpyHostToDevice));
    };
    up(c->d_lin_off, T.lin_off);
    up(c->d_lvl, T.lvl_key);
    up(c->d_bean, T.bean_key);
    up(c->d_irank, T.ident_rank);
    up(c->d_cut, T.cut);
    up(c->d_rcls, T.rank_cls);
    up(c->d_acls, T.allowed_cls);
    up(c->d_linok, T.lin_ok);
    up(c->d_slots, T.slots);
    c->dT.lin_off = c->d_lin_off.p;
    c->dT.lvl_key = c->d_lvl.p;
    c->dT.bean_key = c->d_bean.p;
    c->dT.ident_rank = c->d_irank.p;
    c->dT.cut = c->d_cut.p;
    c->dT.rank_cls = c->d_rcls.p;
    c->dT.allowed_cls = c->d_acls.p;
    c->dT.lin_ok = c->d_linok.p;
    c->dT.slots = c->d_slots.p;
    c->dT.hash_mask = T.hash_mask;
    c->dT.n_lin = (uint32_t)T.n_lin();
}
struct Caps {
    size_t rec, slots, beans, accs, defer, pool;
};

constexpr size_t kIdxMax = 0xFFFFFFF0ull;  // the record fields that index these arrays are 32-bit

// Output capacities for n bytes of text: from the densities learnt on earlier runs / the probe, else from the
// shortest rows the grammar allows for typical BLAST output.  An overflow is counted (never written) by the kernels;
// the host then grows the arrays and runs again.
Caps initial_caps(const blu_ctx* c, uint64_t n, bool want_pool) {
    auto est = [&](double dens, double dflt_div, size_t slack) {
        const double v = dens > 0 ? (double)n * dens * 1.3 : (double)n / dflt_div;
        return (size_t)std::min<double>(v + (double)slack, (double)kIdxMax);
    };
    Caps k;
    k.rec = est(c->dens_rec, 160, 4096);
    k.slots = est(c->dens_slot, 96, 8192 + (size_t)kTileCtasPerSm * (size_t)c->sms * 2048);  // (+ the CTAs' slabs)
    k.beans = est(c->dens_bean, 128, 8192);
    k.accs = est(c->dens_acc, 128, 8192);
    k.defer = std::max<size_t>(k.rec / 8, 65536);
    k.pool = want_pool ? est(c->dens_pool, 24, 65536) : 0;
    return k;
}

inline size_t dup_table_size(const Caps& k) {
    size_t cap = 1024;
    while (cap < 2 * k.rec) cap <<= 1;
    return cap;
}

// `first`: the context also holds what the configurations of a pass share (see Cfg).
void ensure_out(blu_ctx* c, const Caps& k, bool first) {
    if (!c->out) c->out = c->dev_pool->acquire();
    c->out->rec.ensure(k.rec);
    c->out->beans.ensure(k.beans);
    c->out->accs.ensure(k.accs);
    if (k.pool) c->d_pool.ensure(k.pool);
    if (!first) return;
    c->d_top.ensure(k.slots);
    c->d_defer.ensure(k.defer);
    c->d_dup.ensure(dup_table_size(k));
    if (c->keep_hashes) c->d_qhash.ensure(k.rec);
    c->d_big_rows.ensure((size_t)c->sms * kLongTopCap);
    c->d_big_cand.ensure((size_t)c->sms * kLongTopCap);
}

std::string dev_err_message(uint32_t code, uint64_t off) {
    return std::string(dev_err_text(code)) + " (near byte " + std::to_string(off) + " of the blast output)";
}

// `where`: prefix of the message (which configuration of a group failed)
[[noreturn]] void throw_device_error(uint32_t code, uint64_t off, const std::string& where = "") {
    const std::string m = where + dev_err_message(code, off);
    if (code >= DE_INTERNAL) throw std::runtime_error(m);
    if (code >= DE_NUM_UNSUPPORTED) throw UnsupportedErr(m);
    throw DataErr(m);
}

// Grammar-class errors abort the run wherever the row sits (the reference's CSV reader fails on it too).
void check_fatal(const Counters& h, uint64_t stream_base) {
    if (h.err_code) throw_device_error(h.err_code, stream_base + h.err_off);
}

// What a run leaves for its caller to decide on once the duplicate-id check is complete (a multi-device run merges
// the shards' checks first): consensus-class errors are fatal only for a contiguous table.
struct RunStatus {
    uint32_t soft_code = 0;
    uint64_t soft_off = 0;
    bool dup_found = false;
    void note_soft(const Counters& h, uint64_t stream_base) {
        if (h.soft_code && !soft_code) soft_code = h.soft_code, soft_off = stream_base + h.soft_off;
    }
};

// One configuration of a pass over a table: the context whose lineage tables, strategy, output arrays, counters and densities
// its kernels use, the result part it fills, and its capacities, status and last counter snapshot.  A pass has one
// configuration, or several (blu_consensus_run_*_configs) that share what depends on the text only: the tile kernel runs
// once, and the first configuration's context holds the streams, events, text buffers, top-row slots, deferred runs and
// duplicate-id table of the pass.
struct Cfg {
    blu_ctx* c;
    ResultPartOwned* r;
    Caps k{};
    RunStatus st{};
    Counters h{};
};
using Pass = std::vector<Cfg>;

// Records, top-row slots and deferred runs depend on the text only: every configuration of a pass gets the largest capacity
// any of them asks for (the fan-out kernel keeps record indices).  Beans, accession references and the pool are its own.
void share_caps(Pass& g) {
    Caps& k0 = g[0].k;
    for (const Cfg& x : g) k0.rec = std::max(k0.rec, x.k.rec), k0.slots = std::max(k0.slots, x.k.slots), k0.defer = std::max(k0.defer, x.k.defer);
    for (Cfg& x : g) x.k.rec = k0.rec, x.k.slots = k0.slots, x.k.defer = k0.defer;
}

void reset_timings(Pass& g) {
    for (Cfg& x : g) x.c->tm = blu_timings{};
}

// A context of this pass has not seen a table like it yet (see probe_densities).
bool unseen(const Pass& g) {
    for (const Cfg& x : g)
        if (x.c->dens_rec == 0) return true;
    return false;
}

// BLU_SYNC_DEBUG=1: synchronise behind every kernel so that a device fault is attributed to the kernel that caused it
inline void dbg_sync(cudaStream_t s, const char* what) {
    static const bool on = getenv("BLU_SYNC_DEBUG") != nullptr;
    if (!on) return;
    cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

void reset_counters_async(blu_ctx* c, cudaStream_t s) {
    CK(cudaMemsetAsync(c->d_ctr, 0, sizeof(Counters), s));
    CK(cudaMemsetAsync(&c->d_ctr->tail_start, 0xFF, sizeof(unsigned long long), s));
}

// How the strings of a result are delivered.
enum class Strings {
    Pool,      // gathered into a string pool that is downloaded with the records
    DeviceText // references into the device text (device-resident results)
    ,
    HostText   // references into the caller's host text (BLU_OPT_TEXT_REFS): buffer offsets are relocated by `delta`
};

// One range / chunk, all of it queued without a host round trip: tile kernel, long-run kernel (returns at once when
// nothing was deferred), consensus, (gather,) duplicate-id check, and the one-thread kernel that advances the device-side
// cursors and snapshots the counters into mapped host memory.  `begin` may be kBeginFromCounters.
// A pass with several configurations runs the tile kernel once, into the first one's records and counters, and the fan-out
// kernel copies what it found to the others; the long-run, consensus and gather kernels and the advance run per
// configuration, the duplicate-id check once (the others only relocate their references into the caller's text).
void launch_range(const Pass& g, const uint8_t* dtext, uint64_t begin, uint64_t end, bool final_chunk, cudaStream_t s, int slot, Strings strings,
                  long long delta) {
    blu_ctx* c0 = g[0].c;
    const Caps& k0 = g[0].k;
    uint64_t launches = 0;
    auto run_params = [&](const Cfg& x) {
        RunParams p{};
        p.text = dtext;
        p.begin = begin;
        p.end = end;
        p.final_chunk = final_chunk ? 1 : 0;
        p.strategy = x.c->opts.strategy;
        p.T = x.c->dT;
        p.records = x.c->out->rec.p;
        p.rec_cap = x.k.rec;
        p.toprows = c0->d_top.p;
        p.slot_cap = k0.slots;
        p.beans = x.c->out->beans.p;
        p.bean_cap = x.k.beans;
        p.accs = x.c->out->accs.p;
        p.acc_cap = x.k.accs;
        p.defer = c0->d_defer.p;
        p.defer_cap = (uint32_t)std::min<size_t>(k0.defer, 0xFFFFFFFFu);
        p.big_rows = c0->d_big_rows.p;
        p.big_cand = c0->d_big_cand.p;
        p.ctr = x.c->d_ctr;
        return p;
    };
    cudaEvent_t* ev = c0->ev[slot];
    CK(cudaEventRecord(ev[0], s));
    CK(launch_tile_kernel(run_params(g[0]), tile_kernel_grid(c0->device), s));
    dbg_sync(s, "tile_kernel");
    launches++;
    CK(cudaEventRecord(ev[1], s));
    if (g.size() > 1) {
        FanoutParams f{};
        f.src = c0->d_ctr;
        f.src_records = c0->out->rec.p;
        f.n_dst = (int)g.size() - 1;
        f.rec_cap = k0.rec;
        for (size_t i = 1; i < g.size(); i++) f.dst[i - 1] = g[i].c->d_ctr, f.dst_records[i - 1] = g[i].c->out->rec.p;
        CK(launch_fanout_kernel(f, c0->sms, s));
        dbg_sync(s, "fanout_kernel");
        launches++;
    }
    for (const Cfg& x : g) {
        CK(launch_longrun_kernel(run_params(x), c0->sms, s));
        dbg_sync(s, "longrun_kernel");
        launches++;
    }
    CK(cudaEventRecord(ev[2], s));
    for (const Cfg& x : g) {
        PostParams q{};
        q.records = x.c->out->rec.p;
        q.rec_cap = x.k.rec;
        q.toprows = c0->d_top.p;
        q.slot_cap = k0.slots;
        q.beans = x.c->out->beans.p;
        q.bean_cap = x.k.beans;
        q.accs = x.c->out->accs.p;
        q.acc_cap = x.k.accs;
        q.text = dtext;
        q.text_end = end;
        q.pool = strings == Strings::Pool ? x.c->d_pool.p : nullptr;
        q.pool_cap = strings == Strings::Pool ? x.k.pool : 0;
        q.T = x.c->dT;
        q.strategy = x.c->opts.strategy;
        q.ctr = x.c->d_ctr;
        CK(launch_consensus_kernel(q, c0->sms, s));
        dbg_sync(s, "consensus_kernel");
        launches++;
        if (strings == Strings::Pool) {
            CK(launch_gather_kernel(q, c0->sms, s));
            dbg_sync(s, "gather_kernel");
            launches++;
        }
    }
    for (size_t i = 0; i < g.size() && (i == 0 || strings == Strings::HostText); i++) {
        const Cfg& x = g[i];
        DupParams d{};
        d.records = x.c->out->rec.p;
        d.rec_cap = x.k.rec;
        d.beans = x.c->out->beans.p;
        d.accs = x.c->out->accs.p;
        d.strings = strings == Strings::Pool ? x.c->d_pool.p : dtext;
        d.strings_len = strings == Strings::Pool ? x.k.pool : end;
        d.table = i == 0 ? c0->d_dup.p : nullptr;
        d.mask = i == 0 ? (uint32_t)(dup_table_size(k0) - 1) : 0;
        d.hashes = i == 0 && c0->d_qhash.cap >= k0.rec ? c0->d_qhash.p : nullptr;
        d.ref_delta = strings == Strings::HostText ? delta : 0;
        d.ctr = x.c->d_ctr;
        CK(launch_dup_kernel(d, c0->sms, s));
        dbg_sync(s, "dup_kernel");
        launches++;
    }
    for (const Cfg& x : g) {
        AdvanceParams a{};
        a.ctr = x.c->d_ctr;
        a.rec_cap = x.k.rec;
        a.range_end = end;
        a.snapshot = x.c->d_snap + slot;
        CK(launch_advance_kernel(a, s));
        dbg_sync(s, "advance_kernel");
        launches++;
    }
    CK(cudaEventRecord(ev[3], s));
    c0->tm.n_kernel_launches += launches;
}

// Start of a run: output arrays, counters, the duplicate-id table.
void begin_run(const Pass& g, cudaStream_t s) {
    for (size_t i = 0; i < g.size(); i++) {
        ensure_out(g[i].c, g[i].k, i == 0);
        reset_counters_async(g[i].c, s);
    }
    CK(cudaMemsetAsync(g[0].c->d_dup.p, 0, dup_table_size(g[0].k) * sizeof(unsigned long long), s));
}

inline bool overflowed(const Counters& h, const Caps& k) {
    return h.cap_overflow || h.rec_count > k.rec || h.slot_count > k.slots || h.bean_used > k.beans || h.acc_used > k.accs || h.n_defer > k.defer ||
           (k.pool && h.pool_used > k.pool);
}

// `scale` = whole input / part of it the counters cover (>= 1): the cursors are cumulative over the chunks / ranges
// processed so far, so the new capacity is extrapolated to the whole input -- otherwise a table of tiny rows in many
// chunks needs one retry per chunk.  `n_bytes` bounds the extrapolation (a row has >= 26 bytes).
void grow_caps(const Counters& h, Caps& k, double scale, uint64_t n_bytes) {
    bool grew = false;
    scale = std::max(1.0, scale);
    auto want = [&](uint64_t seen, uint64_t slack, uint64_t bound) {
        const double w = (double)seen * scale * 1.125 + (double)slack;
        const double v = std::max<double>((double)seen + (double)slack, std::min<double>(w, (double)bound + (double)slack));
        return (size_t)std::min<double>(v, (double)kIdxMax);
    };
    if (h.rec_count > k.rec) k.rec = want(h.rec_count, 1024, n_bytes / 26), grew = true;
    if (h.slot_count > k.slots) k.slots = want(h.slot_count, 1024, n_bytes / 26 + (1u << 20)), grew = true;
    if (h.bean_used > k.beans) k.beans = want(h.bean_used, 1024, n_bytes / 26), grew = true;
    if (h.acc_used > k.accs) k.accs = want(h.acc_used, 1024, n_bytes / 26), grew = true;
    if (h.n_defer > k.defer) k.defer = (size_t)h.n_defer + h.n_defer / 8 + 1024, grew = true;
    if (k.pool && h.pool_used > k.pool) k.pool = want(h.pool_used, 4096, n_bytes), grew = true;
    if (!grew) {  // overflow flagged but the counts look fine (a reservation raced past the cap): grow everything
        auto dbl = [](size_t v) { return std::min<size_t>(v * 2, kIdxMax); };
        k.rec = dbl(k.rec), k.slots = dbl(k.slots), k.beans = dbl(k.beans), k.accs = dbl(k.accs), k.defer *= 2;
        if (k.pool) k.pool *= 2;
    }
    if (h.rec_count >= kIdxMax || h.slot_count >= kIdxMax || h.bean_used >= kIdxMax || h.acc_used >= kIdxMax)
        throw UnsupportedErr("more than 2^32 queries / top rows in one device's share of the table (shard it over more devices)");
}

void learn_densities(blu_ctx* c, const Counters& h, uint64_t n) {
    if (!n) return;
    c->dens_rec = (double)h.rec_count / (double)n;
    c->dens_slot = (double)h.slot_count / (double)n;
    c->dens_bean = (double)h.bean_used / (double)n;
    c->dens_acc = (double)h.acc_used / (double)n;
    if (h.pool_used) c->dens_pool = (double)h.pool_used / (double)n;
}

// Kernel times of a run, summed over its ranges / chunks.
struct KernelMs {
    double tile = 0, longrun = 0, post = 0;
};

// Reads the counter snapshots of range / chunk `slot` (into Cfg::h) once its kernels have completed: its kernel times and
// deferred runs are added up, a grammar error is raised (at `base` + err_off) before anything is done about a capacity -- a
// malformed row is an error whatever else happened -- and on a capacity overflow of any configuration its capacities are
// grown for the whole input of `n` bytes (`scale`: see grow_caps).  true: the pass has to start over.
bool read_snapshot(Pass& g, int slot, uint64_t base, double scale, uint64_t n, KernelMs& ms) {
    blu_ctx* c0 = g[0].c;
    const cudaEvent_t* ev = c0->ev[slot];
    CK(cudaEventSynchronize(ev[3]));
    for (Cfg& x : g) x.h = x.c->h_snap[slot];
    ms.tile += ev_ms(ev[0], ev[1]);
    ms.longrun += ev_ms(ev[1], ev[2]);
    ms.post += ev_ms(ev[2], ev[3]);
    c0->tm.n_deferred_runs += g[0].h.n_defer;
    for (const Cfg& x : g) check_fatal(x.h, base);
    bool grew = false;
    for (Cfg& x : g)
        if (overflowed(x.h, x.k)) grow_caps(x.h, x.k, scale, n), grew = true;
    if (grew) share_caps(g);
    return grew;
}

// The end of a pass that found no duplicate id (Cfg::h: the last snapshots): the timings every loop reports the same way,
// and the densities that size the next run.
void finish_run(Pass& g, uint64_t n, uint64_t tiles, const KernelMs& ms) {
    if (g[0].h.post_done == 0) throw DataErr("the blast output holds no rows");
    for (const Cfg& x : g) {
        blu_ctx* c = x.c;
        const Counters& h = x.h;
        c->tm.ms_tile_kernel = ms.tile;
        c->tm.ms_longrun_kernel = ms.longrun;
        c->tm.ms_gather_kernel = ms.post;
        c->tm.ms_total_device = ms.tile + ms.longrun + ms.post;
        c->tm.text_bytes = n;
        c->tm.taxonomy_bytes = c->tax->device_bytes();
        c->tm.n_tile_launches = tiles;
        c->tm.n_queries = h.post_done;
        c->tm.n_rows = h.n_rows;
        c->tm.result_bytes = h.post_done * sizeof(blu_record) + h.bean_used * sizeof(blu_bean) + h.acc_used * sizeof(blu_acc);
        c->tm.d2h_bytes += sizeof(Counters);
        learn_densities(c, h, n);
    }
}

// Synchronises the first `n` of `s` when its scope is left by an exception: nothing may still read the caller's text, or a
// buffer that is about to be freed, when the call returns.
struct SyncOnUnwind {
    cudaStream_t s[3];
    int n;
    const int pending = std::uncaught_exceptions();
    ~SyncOnUnwind() {
        if (std::uncaught_exceptions() > pending)
            for (int i = 0; i < n; i++) cudaStreamSynchronize(s[i]);
    }
};

// Incremental download of the finished part of the result arrays on the pass's download stream (that of its first
// context), so that the device->host copies of one range / chunk run under the kernels (and host->device copies) of the
// next one.
struct Downloader {
    blu_ctx* c;
    ResultPartOwned* r;
    cudaStream_t ds;
    uint64_t rec_done = 0, bean_done = 0, acc_done = 0, pool_done = 0;
    uint64_t bytes = 0;

    Downloader(blu_ctx* ctx, ResultPartOwned* res, cudaStream_t stream) : c(ctx), r(res), ds(stream) { r->pinned = c->pool; }

    static void grow(blu_ctx* c, PinnedBuf& b, size_t need, size_t keep, cudaStream_t ds) {
        if (b.cap >= need && b.p) return;
        PinnedBuf nb = c->acquire(std::max<size_t>(need, 64));
        if (keep) {
            CK(cudaStreamSynchronize(ds));  // the prefix may still be in flight
            memcpy(nb.p, b.p, keep);
        }
        if (b.p) c->pool->release(b);
        b = nb;
    }
    // capacity for at least these totals (called with estimates first, exact numbers at the end)
    void reserve(uint64_t rec, uint64_t beans, uint64_t accs, uint64_t pool) {
        grow(c, r->b_rec, rec * sizeof(blu_record), rec_done * sizeof(blu_record), ds);
        grow(c, r->b_beans, beans * sizeof(blu_bean), bean_done * sizeof(blu_bean), ds);
        grow(c, r->b_accs, accs * sizeof(blu_acc), acc_done * sizeof(blu_acc), ds);
        if (pool) grow(c, r->b_pool, pool, pool_done, ds);
    }
    // everything below the cursors of snapshot `h` is final on the device (its post-pass has completed)
    void push(const Counters& h) {
        const uint64_t rec = h.post_done, beans = h.bean_used, accs = h.acc_used, pool = h.pool_used;
        reserve(rec, beans, accs, pool);
        if (rec > rec_done)
            CK(cudaMemcpyAsync((blu_record*)r->b_rec.p + rec_done, c->out->rec.p + rec_done, (rec - rec_done) * sizeof(blu_record), cudaMemcpyDeviceToHost, ds));
        if (beans > bean_done)
            CK(cudaMemcpyAsync((blu_bean*)r->b_beans.p + bean_done, c->out->beans.p + bean_done, (beans - bean_done) * sizeof(blu_bean), cudaMemcpyDeviceToHost, ds));
        if (accs > acc_done)
            CK(cudaMemcpyAsync((blu_acc*)r->b_accs.p + acc_done, c->out->accs.p + acc_done, (accs - acc_done) * sizeof(blu_acc), cudaMemcpyDeviceToHost, ds));
        if (pool > pool_done) CK(cudaMemcpyAsync((char*)r->b_pool.p + pool_done, c->d_pool.p + pool_done, pool - pool_done, cudaMemcpyDeviceToHost, ds));
        bytes += (rec - rec_done) * sizeof(blu_record) + (beans - bean_done) * sizeof(blu_bean) + (accs - acc_done) * sizeof(blu_acc) + (pool - pool_done);
        rec_done = rec, bean_done = beans, acc_done = accs, pool_done = pool;
    }
    void finish(const Counters& h) {
        push(h);
        CK(cudaStreamSynchronize(ds));
        r->n_rec = rec_done, r->n_beans = bean_done, r->n_accs = acc_done, r->pool_len = pool_done;
        r->on_host = true;
        c->tm.d2h_bytes += bytes;
    }
    void abandon() {  // retry with larger device capacities: drop what was downloaded
        cudaStreamSynchronize(ds);
        rec_done = bean_done = acc_done = pool_done = 0;
        bytes = 0;
    }
};

void require_tax(blu_ctx* c) {
    if (!c->tax) throw std::invalid_argument("no taxonomy loaded (call blu_taxonomy_load_json first)");
}

// Output densities of a table this context has not seen the like of: the kernels run once over a small prefix (results
// discarded), so that the arrays of the real run are sized for what the table holds instead of for the shortest rows the
// grammar allows (1.5 GB of records for a 3.8 GB table; more than a B200 has for a 77 GB one).
// A pass with several configurations probes once, for every context that has not seen such a table.
void probe_densities(Pass& g, const uint8_t* dtext, uint64_t begin, uint64_t end, cudaStream_t s) {
    const uint64_t len = end - begin;
    if (len < (1u << 20)) return;
    const blu_timings keep = g[0].c->tm;
    for (Cfg& x : g) x.k = initial_caps(x.c, len, false);
    share_caps(g);
    begin_run(g, s);
    launch_range(g, dtext, begin, end, false, s, 0, Strings::DeviceText, 0);
    CK(cudaEventSynchronize(g[0].c->ev[0][3]));
    g[0].c->tm = keep;
    for (const Cfg& x : g) {
        blu_ctx* c = x.c;
        const Counters h = c->h_snap[0];
        if (c->dens_rec != 0 || overflowed(h, x.k) || h.err_code || h.post_done < 64) continue;  // (the real run reports whatever is wrong)
        const uint64_t covered = h.next_begin > begin && h.next_begin <= end ? h.next_begin - begin : len;
        learn_densities(c, h, covered);
        c->dens_pool = c->dens_rec * 48.0 + c->dens_acc * 24.0;  // (ids + accessions; an underestimate is grown by the retry)
    }
}

struct NonContiguous : std::runtime_error {
    using std::runtime_error::runtime_error;
};

std::vector<uint64_t> resident_ranges(uint64_t n) {
    // Large resident tables are processed in a few query-aligned ranges so that the download of one range's records
    // overlaps the kernels of the next.  Equal ranges measured best (tools/range_split.py, profiles/README.md).
    // BLU_RANGE_FRACS="0.3,0.3,0.25,0.15" overrides the split (measurement knob).
    std::vector<double> fracs(n >= (512ull << 20) ? 4 : (n >= (128ull << 20) ? 2 : 1), 1.0);
    if (const char* ev = getenv("BLU_RANGE_FRACS")) {
        std::vector<double> f;
        for (const char* q = ev; *q;) {
            char* e2 = nullptr;
            double v = strtod(q, &e2);
            if (e2 == q || !(v > 0)) break;
            f.push_back(v);
            q = *e2 == ',' ? e2 + 1 : e2;
        }
        if (!f.empty() && f.size() <= (size_t)kMaxRanges) fracs = f;
    }
    std::vector<uint64_t> range_end(fracs.size());
    double tot = 0, acc = 0;
    for (double f : fracs) tot += f;
    for (size_t i = 0; i < fracs.size(); i++) {
        acc += fracs[i];
        const uint64_t e = (uint64_t)((double)n * (acc / tot));
        range_end[i] = std::min<uint64_t>(n, (e + (uint64_t)kTile - 1) / (uint64_t)kTile * (uint64_t)kTile);
    }
    range_end.back() = n;
    return range_end;
}

void check_device_text(const uint8_t* dtext, uint64_t n) {
    if (n == 0) throw DataErr("empty blast output (the reference's CsvReader fails on an empty file)");
    if (((uintptr_t)dtext & 15) != 0) throw std::invalid_argument("device text must be 16-byte aligned");
}

// --- text resident on the device ------------------------------------------------------------------------------------
// resident: one range, five launches, one host synchronisation; nothing but the counters crosses PCIe and the result keeps
// the device arrays and references into the device text (SURVEY 8d(i)).
// Otherwise the result is downloaded: every range's kernels are queued up front -- a range starts where the previous one
// stopped (Counters.next_begin), the post-pass takes its record range from the device counters -- so the GPU never waits
// for the host; the host trails behind, reads each range's snapshot when its event fires and queues that range's download
// on the download stream.
void run_device_text(Pass& g, const uint8_t* dtext, uint64_t n, cudaStream_t s, bool resident) {
    blu_ctx* c0 = g[0].c;
    SyncOnUnwind unwind{{s, c0->d2h_stream}, resident ? 1 : 2};
    for (const Cfg& x : g) require_tax(x.c);
    check_device_text(dtext, n);
    reset_timings(g);
    if (unseen(g) && n > (64ull << 20)) probe_densities(g, dtext, 0, std::min<uint64_t>(n, 32ull << 20), s);
    for (Cfg& x : g) x.k = initial_caps(x.c, n, !resident);
    share_caps(g);
    const std::vector<uint64_t> range_end = resident ? std::vector<uint64_t>{n} : resident_ranges(n);
    const int n_ranges = (int)range_end.size();
    const Strings strings = resident ? Strings::DeviceText : Strings::Pool;
    std::vector<Downloader> dl;
    for (const Cfg& x : g) dl.emplace_back(x.c, x.r, c0->d2h_stream);
    for (int attempt = 0; attempt < 8; attempt++) {
        begin_run(g, s);
        for (int ri = 0; ri < n_ranges; ri++)
            launch_range(g, dtext, ri == 0 ? 0 : kBeginFromCounters, range_end[ri], ri + 1 == n_ranges, s, ri, strings, 0);
        bool retry = false;
        KernelMs ms;
        for (int ri = 0; ri < n_ranges && !retry; ri++) {
            retry = read_snapshot(g, ri, 0, (double)n / (double)std::max<uint64_t>(range_end[ri], 1), n, ms);
            if (!retry && ri + 1 < n_ranges && !g[0].h.dup_found)
                for (size_t i = 0; i < g.size(); i++) {
                    const Counters& h = g[i].h;
                    if (ri == 0 && range_end[0] > 0) {
                        // size the pinned result buffers from the density of the first range
                        const double f = 1.15 * (double)n / (double)range_end[0];
                        dl[i].reserve((uint64_t)(h.post_done * f) + 4096, (uint64_t)(h.bean_used * f) + 8192, (uint64_t)(h.acc_used * f) + 8192,
                                      (uint64_t)(h.pool_used * f) + 65536);
                    }
                    dl[i].push(h);  // runs on the download stream under the next ranges' kernels
                }
        }
        if (retry) {
            if (!resident) {
                CK(cudaStreamSynchronize(s));  // the later ranges are still queued
                for (Downloader& d : dl) d.abandon();
            }
            reset_timings(g);
            continue;
        }
        for (Cfg& x : g) {
            x.st.note_soft(x.h, 0);
            x.st.dup_found = g[0].h.dup_found != 0;
        }
        if (g[0].st.dup_found) {
            if (!resident)
                for (Downloader& d : dl) d.abandon();
            return;
        }
        finish_run(g, n, (uint64_t)n_ranges, ms);
        for (size_t i = 0; i < g.size(); i++) {
            const Counters& h = g[i].h;
            if (!resident) {
                dl[i].finish(h);
                continue;
            }
            blu_ctx* c = g[i].c;
            ResultPartOwned* r = g[i].r;
            r->dev = std::move(c->out);
            r->dev_pool = c->dev_pool;
            r->ctx = c;
            r->dtext = dtext;
            r->dtext_len = n;
            r->n_rec = h.post_done, r->n_beans = h.bean_used, r->n_accs = h.acc_used;
            r->on_host = false;
        }
        return;
    }
    throw std::runtime_error("output capacity did not converge");
}

// Brings a device-resident part to the host: the referenced strings are gathered into a pool first (a counting pass of
// the gather kernel sizes it), then records, beans, accession references and the pool are downloaded.
void download_part(ResultPartOwned* r) {
    if (r->on_host) return;
    blu_ctx* c = r->ctx;
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    PostParams q{};
    q.records = r->dev->rec.p;
    q.rec_cap = r->n_rec;
    q.beans = r->dev->beans.p;
    q.bean_cap = r->n_beans;
    q.accs = r->dev->accs.p;
    q.acc_cap = r->n_accs;
    q.text = r->dtext;
    q.text_end = r->dtext_len;
    q.ctr = c->d_ctr;
    Counters hc{};
    hc.rec_count = r->n_rec;
    hc.tail_start = ~0ull;
    CK(cudaMemcpyAsync(c->d_ctr, &hc, sizeof hc, cudaMemcpyHostToDevice, s));
    q.pool = nullptr;  // counting pass
    CK(launch_gather_kernel(q, c->sms, s));
    Counters got{};
    CK(cudaMemcpyAsync(&got, c->d_ctr, sizeof got, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const uint64_t pool_len = got.pool_used;
    c->d_pool.ensure(std::max<uint64_t>(pool_len, 64));
    CK(cudaMemcpyAsync(c->d_ctr, &hc, sizeof hc, cudaMemcpyHostToDevice, s));
    q.pool = c->d_pool.p;
    q.pool_cap = pool_len;
    CK(launch_gather_kernel(q, c->sms, s));
    r->pinned = c->pool;
    r->b_rec = c->acquire(std::max<uint64_t>(r->n_rec * sizeof(blu_record), 64));
    r->b_beans = c->acquire(std::max<uint64_t>(r->n_beans * sizeof(blu_bean), 64));
    r->b_accs = c->acquire(std::max<uint64_t>(r->n_accs * sizeof(blu_acc), 64));
    r->b_pool = c->acquire(std::max<uint64_t>(pool_len, 64));
    if (r->n_rec) CK(cudaMemcpyAsync(r->b_rec.p, r->dev->rec.p, r->n_rec * sizeof(blu_record), cudaMemcpyDeviceToHost, s));
    if (r->n_beans) CK(cudaMemcpyAsync(r->b_beans.p, r->dev->beans.p, r->n_beans * sizeof(blu_bean), cudaMemcpyDeviceToHost, s));
    if (r->n_accs) CK(cudaMemcpyAsync(r->b_accs.p, r->dev->accs.p, r->n_accs * sizeof(blu_acc), cudaMemcpyDeviceToHost, s));
    if (pool_len) CK(cudaMemcpyAsync(r->b_pool.p, c->d_pool.p, pool_len, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&got, c->d_ctr, sizeof got, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (got.cap_overflow) throw std::runtime_error("string pool of a device-resident result did not fit its counted size");
    r->pool_len = pool_len;
    r->dev_pool->release(std::move(r->dev));
    r->on_host = true;
}


// Non-contiguous hit tables (the reference groups rows through a HashMap<String, Vec<_>>, mod.rs:145,192, so the
// rows of one query need not be adjacent).  Rare (BLAST emits queries contiguously, blutils appends whole chunks),
// so it is handled by data movement only: rows are regrouped by query id -- first-appearance order of the queries,
// file order inside a query, which is all the consensus depends on -- and the GPU pipeline runs on the regrouped
// text.  No consensus arithmetic happens on the host.
std::string regroup_by_query(const char* text, uint64_t n) {
    struct Row {
        uint64_t off;
        uint32_t len;
    };
    std::unordered_map<std::string_view, uint32_t> gid;
    std::vector<std::vector<Row>> groups;
    for (uint64_t p = 0; p < n;) {
        const char* nl = (const char*)memchr(text + p, '\n', n - p);
        const uint64_t e = nl ? (uint64_t)(nl - text) : n;
        if (e > p) {
            const char* tab = (const char*)memchr(text + p, '\t', e - p);
            std::string_view q(text + p, tab ? (size_t)(tab - (text + p)) : (size_t)(e - p));
            auto it = gid.find(q);
            uint32_t g;
            if (it == gid.end()) {
                g = (uint32_t)groups.size();
                gid.emplace(q, g);
                groups.emplace_back();
            } else
                g = it->second;
            groups[g].push_back({p, (uint32_t)(e - p)});
        }
        p = e + 1;
    }
    std::string out;
    out.reserve(n + 1);
    for (auto& g : groups)
        for (auto& r : g) {
            out.append(text + r.off, r.len);
            out.push_back('\n');
        }
    return out;
}

// The same regrouping on the GPU (blu_regroup.cu): the table -- uploaded first when it is host text -- is rewritten in HBM.
// Used whenever the table, its regrouped copy and ~72 bytes per row fit the device; BLU_REGROUP_HOST=1 forces the host path.
bool regroup_gpu(blu_ctx* c, const char* h_text, const uint8_t* d_text, uint64_t n, cudaStream_t s, DevMem& out) {
    if (const char* ev = getenv("BLU_REGROUP_HOST"))
        if (atoi(ev)) return false;
    if (n == 0) return false;
    if (c->is_multi()) {  // on the context's first GPU, with that shard's stream
        c = c->shards[0].get();
        s = c->stream;
    }
    CK(cudaSetDevice(c->device));
    DevMem in;
    const auto t0 = std::chrono::steady_clock::now();
    if (!d_text) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        if (2.2 * (double)n + (double)(256ull << 20) > (double)free_b) return false;
        if (!in.alloc(n + 512)) return false;
        CK(cudaMemcpyAsync(in.p, h_text, n, cudaMemcpyHostToDevice, s));
        d_text = in.p;
    }
    uint64_t rows = 0;
    const bool trace = getenv("BLU_REGROUP_TRACE") != nullptr;
    if (trace) cudaStreamSynchronize(s);
    const auto t1 = std::chrono::steady_clock::now();
    const int rc = regroup_device(d_text, n, s, &out.p, &out.n, &rows);
    if (trace)
        fprintf(stderr, "[blu regroup] upload %.2f ms, regroup_device %.2f ms (%llu rows, rc %d)\n", std::chrono::duration<double, std::milli>(t1 - t0).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count(), (unsigned long long)rows, rc);
    if (rc < 0) throw CudaErr(std::string("regroup_device: ") + cudaGetErrorString((cudaError_t)(-rc)));
    return rc == 0;
}

// --- where the streamed path takes the text of chunk `ci` from -------------------------------------------------
struct ChunkSource {
    virtual ~ChunkSource() = default;
    virtual const char* acquire(uint64_t ci) = 0;  // host pointer to chunk ci (may block until it is there)
    virtual void release(uint64_t) {}              // the host->device copy of chunk ci has completed
    virtual void restart() {}                      // the run starts over from chunk 0 (no copy is in flight)
};

struct MemorySource : ChunkSource {
    const char* text;
    uint64_t chunk;
    MemorySource(const char* t, uint64_t ch) : text(t), chunk(ch) {}
    const char* acquire(uint64_t ci) override { return text + ci * chunk; }
};

// A file, read by parallel pread()s into a ring of three pinned staging buffers while earlier chunks are copied to
// the device and processed: the file never has to fit in (pinned) host memory, and reading overlaps everything else.
class FileSource : public ChunkSource {
    static constexpr uint64_t kRing = 3;
    blu_ctx* c_;
    int fd_;
    uint64_t base_, n_, chunk_, n_chunks_;  // the source is bytes [base_, base_ + n_) of the file
    int n_readers_;
    PinnedBuf buf_[kRing];
    std::mutex mu_;
    std::condition_variable cv_;
    uint64_t staged_ = 0;    // chunks [0, staged_) of this epoch are in their buffers
    uint64_t released_ = 0;  // chunks [0, released_) may be overwritten
    uint64_t epoch_ = 0;
    bool stop_ = false;
    std::string error_;
    std::thread coordinator_;
    bool read_span(char* dst, uint64_t off, uint64_t len, std::string& err) const {
        while (len) {
            ssize_t got = pread(fd_, dst, (size_t)std::min<uint64_t>(len, 1ull << 30), (off_t)(base_ + off));
            if (got < 0 && errno == EINTR) continue;
            if (got <= 0) {
                err = got == 0 ? "the blast output shrank while it was read" : std::string("read error on the blast output: ") + strerror(errno);
                return false;
            }
            dst += got, off += (uint64_t)got, len -= (uint64_t)got;
        }
        return true;
    }
    bool read_chunk(uint64_t ci, std::string& err) const {
        char* dst = (char*)buf_[ci % kRing].p;
        const uint64_t off = ci * chunk_, len = std::min(chunk_, n_ - off);
        const uint64_t slice = std::max<uint64_t>(((len + n_readers_ - 1) / n_readers_ + 4095) & ~4095ull, 1ull << 20);
        std::vector<std::thread> th;
        std::vector<std::string> errs((size_t)n_readers_);
        std::atomic<bool> ok{true};
        int t = 0;
        try {
            for (uint64_t o = slice; o < len; o += slice, t++)
                th.emplace_back([&, o, t] {
                    if (!read_span(dst + o, off + o, std::min(slice, len - o), errs[(size_t)t])) ok = false;
                });
        } catch (...) {  // could not start a thread: the ones already running must be joined before unwinding
            for (auto& x : th) x.join();
            throw;
        }
        std::string e0;
        if (!read_span(dst, off, std::min(slice, len), e0)) ok = false;
        for (auto& x : th) x.join();
        if (!ok) {
            err = e0;
            for (auto& e : errs)
                if (err.empty()) err = e;
        }
        return ok;
    }
    void run() {
        uint64_t my_epoch = 0, next = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || epoch_ != my_epoch || (next < n_chunks_ && next < released_ + kRing); });
                if (stop_) return;
                if (epoch_ != my_epoch) {
                    my_epoch = epoch_, next = 0;
                    continue;
                }
            }
            std::string err;
            bool ok = false;
            try {
                ok = read_chunk(next, err);
            } catch (const std::exception& e) {  // e.g. no more threads: reported through acquire(), not std::terminate
                err = std::string("reading the blast output failed: ") + e.what();
            }
            {
                std::lock_guard<std::mutex> g(mu_);
                if (epoch_ == my_epoch) {
                    if (ok)
                        staged_ = next + 1;
                    else
                        error_ = err;
                }
            }
            cv_.notify_all();
            next = ok ? next + 1 : n_chunks_;  // after an error: idle until restart() or the destructor
        }
    }

   public:
    FileSource(blu_ctx* c, int fd, uint64_t base, uint64_t n, uint64_t chunk, int sharers = 1)
        : c_(c), fd_(fd), base_(base), n_(n), chunk_(chunk), n_chunks_((n + chunk - 1) / chunk) {
        // readers: the page-cache copy is the bound of this path (DESIGN.md), one thread moves ~5.6 GB/s; `sharers` = the
        // file sources of a multi-device run that share the host's cores.  (Measured and dropped: the file mmap'ed and copied
        // into the ring with memcpy -- 26 / 29 GB/s with 8 / 16 threads against 30 / 39 GB/s for pread.)
        const unsigned hc = std::thread::hardware_concurrency();
        n_readers_ = (int)std::min<unsigned>(16, std::max<unsigned>(2, (hc ? hc : 8) / (unsigned)std::max(1, sharers)));
        if (const char* ev = getenv("BLU_READ_THREADS")) n_readers_ = std::max(1, std::min(64, atoi(ev)));
        const uint64_t used = std::min<uint64_t>(kRing, n_chunks_);
        try {
            for (uint64_t i = 0; i < used; i++) buf_[i] = c->acquire(std::min(chunk, n));
            coordinator_ = std::thread([this] { run(); });
        } catch (...) {  // a constructor that throws gets no destructor call
            for (auto& b : buf_) c_->pool->release(b);
            throw;
        }
    }
    ~FileSource() override {
        {
            std::lock_guard<std::mutex> g(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        coordinator_.join();
        for (auto& b : buf_) c_->pool->release(b);
    }
    const char* acquire(uint64_t ci) override {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return staged_ > ci || !error_.empty(); });
        if (staged_ <= ci) throw IoErr(error_);
        return (const char*)buf_[ci % kRing].p;
    }
    void release(uint64_t ci) override {
        {
            std::lock_guard<std::mutex> g(mu_);
            released_ = std::max(released_, ci + 1);
        }
        cv_.notify_all();
    }
    void restart() override {
        {
            std::lock_guard<std::mutex> g(mu_);
            epoch_++;
            staged_ = released_ = 0;
            error_.clear();
        }
        cv_.notify_all();
    }
};

// --- text on the host: chunked, double-buffered H2D overlapped with the kernels --------------------------------
inline uint64_t chunk_bytes_of(const blu_ctx* c, uint64_t dflt) { return c->opts.chunk_bytes ? ((c->opts.chunk_bytes + 127) & ~127ull) : dflt; }

// `host_text` != nullptr: BLU_OPT_TEXT_REFS -- the result's strings stay references into that (caller-owned) text.
// Several configurations share the chunks: each crosses PCIe once, into the first context's buffers.
void run_host_chunks(Pass& g, ChunkSource& src, uint64_t n, const uint64_t chunk, const char* host_text) {
    blu_ctx* c = g[0].c;
    SyncOnUnwind unwind{{c->copy_stream, c->stream, c->d2h_stream}, 3};  // (and nothing may still copy from a staging buffer)
    for (const Cfg& x : g) require_tax(x.c);
    if (n == 0) throw DataErr("empty blast output (the reference's CsvReader fails on an empty file)");
    reset_timings(g);
    const uint64_t carry = c->carry_bytes;
    const uint64_t n_chunks = (n + chunk - 1) / chunk;
    const bool single = n_chunks == 1;
    const uint64_t buf_bytes = (single ? 0 : carry) + std::min(chunk, n) + 256;
    const uint64_t text_off = single ? 0 : carry;  // where H2D data lands inside a buffer
    c->d_text[0].ensure(buf_bytes);
    if (!single) c->d_text[1].ensure(buf_bytes);
    const Strings strings = host_text ? Strings::HostText : Strings::Pool;
    cudaStream_t s = c->stream, cs = c->copy_stream;
    std::vector<Downloader> dl;
    for (const Cfg& x : g) dl.emplace_back(x.c, x.r, c->d2h_stream);
    auto t0 = std::chrono::steady_clock::now();
    bool have_caps = false;
    for (int attempt = 0; attempt < 8; attempt++) {
        bool retry = false;
        uint64_t tail_len = 0;  // bytes carried from the previous chunk
        KernelMs ms;
        auto issue_h2d = [&](uint64_t ci) {
            const uint64_t off = ci * chunk, len = std::min(chunk, n - off);
            CK(cudaMemcpyAsync(c->d_text[ci & 1].p + text_off, src.acquire(ci), len, cudaMemcpyHostToDevice, cs));
            CK(cudaEventRecord(c->ev_h2d[ci & 1], cs));
            c->tm.h2d_bytes += len;
        };
        issue_h2d(0);
        if (!have_caps) {
            // a table this context has not seen the like of: the first chunk's first megabytes tell how dense its output is
            if (unseen(g) && n > (64ull << 20)) {
                CK(cudaStreamWaitEvent(s, c->ev_h2d[0], 0));
                probe_densities(g, c->d_text[0].p, text_off, text_off + std::min<uint64_t>(std::min(chunk, n), 32ull << 20), s);
            }
            for (Cfg& x : g) x.k = initial_caps(x.c, n, strings == Strings::Pool);
            share_caps(g);
            have_caps = true;
        }
        begin_run(g, s);
        for (uint64_t ci = 0; ci < n_chunks; ci++) {
            const uint64_t off = ci * chunk, len = std::min(chunk, n - off);
            const bool final_chunk = ci + 1 == n_chunks;
            const int slot = (int)(ci % kMaxRanges);
            uint8_t* buf = c->d_text[ci & 1].p;
            CK(cudaStreamWaitEvent(s, c->ev_h2d[ci & 1], 0));
            if (tail_len) {
                // the unfinished last query of the previous chunk goes in front of this chunk's text
                const uint8_t* prev = c->d_text[(ci - 1) & 1].p;
                const uint64_t prev_end = text_off + std::min(chunk, n - (ci - 1) * chunk);
                CK(cudaMemcpyAsync(buf + text_off - tail_len, prev + prev_end - tail_len, tail_len, cudaMemcpyDeviceToDevice, s));
            }
            CK(cudaEventRecord(c->ev_free[(ci + 1) & 1], s));  // previous buffer no longer read after this point
            const uint64_t begin = text_off - tail_len, end = text_off + len;
            // buffer offset d of this chunk is byte off + d - text_off of the caller's text
            launch_range(g, buf, begin, end, final_chunk, s, slot, strings, (long long)off - (long long)text_off);
            if (!final_chunk) {  // behind the launches: a file source may block here until the next chunk has been read
                CK(cudaStreamWaitEvent(cs, c->ev_free[(ci + 1) & 1], 0));
                issue_h2d(ci + 1);
            }
            retry = read_snapshot(g, slot, off - text_off, (double)n / (double)(off + len), n, ms);  // err_off is in buffer coordinates
            src.release(ci);  // `s` waited for this chunk's copy, so it has completed
            if (retry) break;
            for (Cfg& x : g) x.st.note_soft(x.h, off - text_off);
            if (!final_chunk) {
                tail_len = end - g[0].h.next_begin;  // (next_begin == end: nothing is carried)
                if (tail_len > carry) throw UnsupportedErr("a single query spans more than the 64 MiB carry buffer between streamed chunks");
                if (!g[0].h.dup_found)
                    for (size_t i = 0; i < g.size(); i++) {
                        const Counters& h = g[i].h;
                        if (ci == 0) {
                            const double f = 1.15 * (double)n / (double)len;
                            dl[i].reserve((uint64_t)(h.post_done * f) + 4096, (uint64_t)(h.bean_used * f) + 8192, (uint64_t)(h.acc_used * f) + 8192,
                                          strings == Strings::Pool ? (uint64_t)(h.pool_used * f) + 65536 : 0);
                        }
                        dl[i].push(h);  // result download of this chunk runs beside the next chunks' host->device copies
                    }
            }
        }
        if (retry) {
            CK(cudaStreamSynchronize(cs));
            CK(cudaStreamSynchronize(s));
            for (Downloader& d : dl) d.abandon();
            src.restart();
            reset_timings(g);
            for (Cfg& x : g) x.st = RunStatus{};
            continue;
        }
        for (Cfg& x : g) x.st.dup_found = g[0].h.dup_found != 0;
        if (g[0].st.dup_found) {
            for (Downloader& d : dl) d.abandon();
            return;
        }
        finish_run(g, n, n_chunks, ms);
        for (size_t i = 0; i < g.size(); i++) {
            dl[i].finish(g[i].h);
            if (host_text) g[i].r->ext_strings = host_text, g[i].r->ext_len = n;
        }
        c->tm.ms_total_device = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        return;
    }
    throw std::runtime_error("output capacity did not converge");
}

// ---- sharding (SURVEY 8e) ---------------------------------------------------------------------------------------
// Byte access to a table that is either in memory or a file (read through a small window cache): the cut search only
// ever looks at a few rows around each cut.
struct ByteView {
    const char* mem = nullptr;
    int fd = -1;
    uint64_t n = 0;
    ByteView(const char* text, uint64_t len) : mem(text), n(len) {}
    ByteView(int file, uint64_t len) : fd(file), n(len) {}
    mutable std::vector<char> win;
    mutable uint64_t win_lo = 0, win_hi = 0;
    char at(uint64_t i) const {
        if (mem) return mem[i];
        if (i < win_lo || i >= win_hi) {
            const uint64_t lo = i & ~((1ull << 16) - 1);
            const uint64_t len = std::min<uint64_t>(1ull << 20, n - lo);
            win.resize((size_t)len);
            uint64_t got_total = 0;
            while (got_total < len) {
                ssize_t got = pread(fd, win.data() + got_total, (size_t)(len - got_total), (off_t)(lo + got_total));
                if (got < 0 && errno == EINTR) continue;
                if (got <= 0) throw IoErr("Unexpected error occurred on load table.");
                got_total += (uint64_t)got;
            }
            win_lo = lo, win_hi = lo + len;
        }
        return win[(size_t)(i - win_lo)];
    }
};

// cuts[0..n_shards]: ranges of roughly equal size that never split a query (every cut moves forward to the next query
// boundary).  Valid for contiguous tables; a scattered table is caught by the duplicate-id check afterwards.
void shard_cuts(const ByteView& v, int n_shards, uint64_t* cuts) {
    const uint64_t n = v.n;
    auto row_end = [&](uint64_t p) {  // position of the newline that ends the row containing p, or n
        while (p < n && v.at(p) != '\n') p++;
        return p;
    };
    auto next_row = [&](uint64_t p) {  // start of the next non-empty row after the row containing p
        uint64_t q = row_end(p);
        while (q < n && v.at(q) == '\n') q++;
        return q;
    };
    auto first_field = [&](uint64_t a) {  // (copied out: the view of a file keeps one window, and the rows compared with it lie ahead)
        std::string f;
        for (uint64_t i = a; i < n; i++) {
            const char ch = v.at(i);
            if (ch == '\t' || ch == '\n') break;
            f.push_back(ch);
        }
        return f;
    };
    auto has_first_field = [&](uint64_t b, const std::string& f) {
        for (size_t i = 0; i < f.size(); i++)
            if (b + i >= n || v.at(b + i) != f[i]) return false;
        const uint64_t e = b + f.size();
        return e >= n || v.at(e) == '\t' || v.at(e) == '\n';
    };
    cuts[0] = 0;
    cuts[n_shards] = n;
    for (int k = 1; k < n_shards; k++) {
        uint64_t p = std::max<uint64_t>(cuts[k - 1], n / (uint64_t)n_shards * (uint64_t)k);
        if (p >= n) {
            cuts[k] = n;
            continue;
        }
        // first row start at/after p
        if (p > 0 && v.at(p - 1) != '\n') p = next_row(p);
        while (p < n && v.at(p) == '\n') p++;
        if (p >= n) {
            cuts[k] = n;
            continue;
        }
        // previous non-empty row
        if (p > 0) {
            uint64_t q = p - 1;
            while (q > 0 && v.at(q) == '\n') q--;
            if (v.at(q) != '\n') {
                uint64_t st = q;
                while (st > 0 && v.at(st - 1) != '\n') st--;
                const std::string run = first_field(st);
                while (p < n && has_first_field(p, run)) p = next_row(p);  // never split a query
            }
        }
        cuts[k] = p;
    }
}

// ---- one table over several GPUs ---------------------------------------------------------------------------------------
// Cross-shard duplicate-id check: the 64-bit id hashes every shard's duplicate kernel left behind are copied to the first
// device and inserted into one table there (8 bytes per query; the only data that ever moves between the GPUs).
bool merged_duplicate_check(blu_ctx* c, const std::vector<uint64_t>& n_rec) {
    uint64_t total = 0;
    for (uint64_t v : n_rec) total += v;
    if (total == 0) return false;
    blu_ctx* c0 = c->shards[0].get();
    CK(cudaSetDevice(c0->device));
    DevBuf<unsigned long long> all, table;
    struct Cleanup {
        DevBuf<unsigned long long>&a, &b;
        ~Cleanup() { a.release(), b.release(); }
    } cleanup{all, table};
    all.ensure(total);
    size_t cap = 1024;
    while (cap < 2 * total) cap <<= 1;
    table.ensure(cap + 1);  // (+1: the flag)
    CK(cudaMemsetAsync(table.p, 0, (cap + 1) * sizeof(unsigned long long), c0->stream));
    uint64_t at = 0;
    for (size_t i = 0; i < c->shards.size(); i++) {
        if (!n_rec[i]) continue;
        CK(cudaMemcpyPeerAsync(all.p + at, c0->device, c->shards[i]->d_qhash.p, c->shards[i]->device, n_rec[i] * sizeof(unsigned long long), c0->stream));
        at += n_rec[i];
    }
    unsigned int* flag = reinterpret_cast<unsigned int*>(table.p + cap);
    CK(launch_dup_merge_kernel(all.p, total, table.p, (uint32_t)(cap - 1), flag, c0->sms, c0->stream));
    unsigned int found = 0;
    CK(cudaMemcpyAsync(&found, flag, sizeof found, cudaMemcpyDeviceToHost, c0->stream));
    CK(cudaStreamSynchronize(c0->stream));
    return found != 0;
}

// Runs `work(i)` for every shard on its own host thread (each binds its GPU), rethrows the first failure in shard order.
template <class F>
void for_each_shard(blu_ctx* c, F&& work) {
    const size_t N = c->shards.size();
    std::vector<std::exception_ptr> errs(N);
    std::vector<std::thread> th;
    for (size_t i = 0; i < N; i++)
        th.emplace_back([&, i] {
            try {
                if (cudaSetDevice(c->shards[i]->device) != cudaSuccess) throw CudaErr("cudaSetDevice failed");
                work(i);
            } catch (...) {
                errs[i] = std::current_exception();
            }
        });
    for (auto& t : th) t.join();
    for (auto& e : errs)
        if (e) std::rethrow_exception(e);
}

void aggregate_timings(blu_ctx* c, uint64_t n, double wall_ms) {
    blu_timings t{};
    for (auto& sh : c->shards) {
        const blu_timings& u = sh->tm;
        t.ms_tile_kernel = std::max(t.ms_tile_kernel, u.ms_tile_kernel);
        t.ms_longrun_kernel = std::max(t.ms_longrun_kernel, u.ms_longrun_kernel);
        t.ms_gather_kernel = std::max(t.ms_gather_kernel, u.ms_gather_kernel);
        t.result_bytes += u.result_bytes;
        t.taxonomy_bytes += u.taxonomy_bytes;
        t.h2d_bytes += u.h2d_bytes, t.d2h_bytes += u.d2h_bytes;
        t.n_queries += u.n_queries, t.n_rows += u.n_rows, t.n_deferred_runs += u.n_deferred_runs;
        t.n_kernel_launches += u.n_kernel_launches;
        t.n_tile_launches = std::max(t.n_tile_launches, u.n_tile_launches);
    }
    t.text_bytes = n;
    t.ms_total_device = wall_ms;
    c->tm = t;
}

// After all shards have run: the cross-shard duplicate check, then (for a contiguous table) the consensus-class errors.
void settle_multi(blu_ctx* c, const std::vector<RunStatus>& st, const uint64_t* cuts, const std::vector<uint64_t>& n_rec) {
    bool dup = false;
    for (auto& s : st) dup |= s.dup_found;
    if (!dup) dup = merged_duplicate_check(c, n_rec);
    if (dup) throw NonContiguous("a query id occurs in two non-adjacent groups of rows");
    for (size_t i = 0; i < st.size(); i++)
        if (st[i].soft_code) throw_device_error(st[i].soft_code, cuts[i] + st[i].soft_off);
}

// Drops what a result holds and gives it n empty parts.
void reset_parts(blu_result* r, size_t n) {
    for (auto& p : r->parts) p.free_buffers();
    r->parts.clear();
    r->parts.resize(n);
}

// Bytes [begin, begin + len) of a table in memory or in a file through the host-text loop of single-device contexts.
// `sharers`: the file sources of a multi-device run that share the host's cores.
void run_span(Pass& g, const ByteView& v, uint64_t begin, uint64_t len, bool text_refs, int sharers) {
    blu_ctx* c = g[0].c;
    if (v.mem) {
        const uint64_t chunk = chunk_bytes_of(c, 256ull << 20);
        MemorySource src(v.mem + begin, chunk);
        run_host_chunks(g, src, len, chunk, text_refs ? v.mem + begin : nullptr);
    } else {
        const uint64_t chunk = chunk_bytes_of(c, 64ull << 20);
        FileSource src(c, v.fd, begin, len, chunk, sharers);
        run_host_chunks(g, src, len, chunk, nullptr);
    }
}

// One table over the GPUs of a multi-device context: cut at query boundaries, each shard run on its own host thread.
void run_sharded(blu_ctx* c, const ByteView& v, blu_result* r, bool text_refs) {
    if (v.n == 0) throw DataErr("empty blast output (the reference's CsvReader fails on an empty file)");
    const size_t N = c->shards.size();
    std::vector<uint64_t> cuts(N + 1);
    shard_cuts(v, (int)N, cuts.data());
    reset_parts(r, N);
    std::vector<RunStatus> st(N);
    auto t0 = std::chrono::steady_clock::now();
    for_each_shard(c, [&](size_t i) {
        blu_ctx* sh = c->shards[i].get();
        sh->tm = blu_timings{};
        if (cuts[i + 1] <= cuts[i]) return;
        Pass g{Cfg{sh, &r->parts[i]}};
        run_span(g, v, cuts[i], cuts[i + 1] - cuts[i], text_refs, (int)N);
        st[i] = g[0].st;
    });
    std::vector<uint64_t> n_rec(N);
    for (size_t i = 0; i < N; i++) n_rec[i] = st[i].dup_found ? 0 : r->parts[i].n_rec;
    settle_multi(c, st, cuts.data(), n_rec);
    aggregate_timings(c, v.n, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    r->n_rows = c->tm.n_rows;
}

// The configurations of one call and the results they fill: one for blu_consensus_run_*, up to kMaxConfigs single-device
// contexts of one GPU for blu_consensus_run_*_configs.
struct Member {
    blu_ctx* c;
    blu_result* r;
};
using Group = std::vector<Member>;

// A single-device pass over the group: every result gets one empty part.
Pass new_pass(const Group& g) {
    Pass p;
    for (const Member& m : g) {
        reset_parts(m.r, 1);
        p.push_back(Cfg{m.c, &m.r->parts[0]});
    }
    return p;
}

// What a single-device pass leaves for its caller: a repeated id (the table is regrouped and run again), else the
// consensus-class error of the lowest configuration that has one -- named by its index when the pass has several.
void settle(const Group& g, const Pass& p) {
    if (p[0].st.dup_found) throw NonContiguous("a query id occurs in two non-adjacent groups of rows");
    for (size_t i = 0; i < p.size(); i++)
        if (p[i].st.soft_code) throw_device_error(p[i].st.soft_code, p[i].st.soft_off, p.size() > 1 ? "ctxs[" + std::to_string(i) + "]: " : "");
    for (const Member& m : g) m.r->n_rows = m.c->tm.n_rows;
}

// A table in host memory or a file -> results, on one or several GPUs (a group has one context then).  `text_refs` applies
// to host memory only.
void run_table(const Group& g, const ByteView& v, bool text_refs) {
    blu_ctx* c = g[0].c;
    if (c->is_multi()) {
        run_sharded(c, v, g[0].r, text_refs);
        return;
    }
    CK(cudaSetDevice(c->device));
    Pass p = new_pass(g);
    run_span(p, v, 0, v.n, text_refs, 1);
    settle(g, p);
}

// The regrouped table (device memory of ours) through the device-text loop of single-device contexts.
void run_regrouped_device(const Group& g, const DevMem& dt, cudaStream_t s, bool resident) {
    Pass p = new_pass(g);
    run_device_text(p, dt.p, dt.n, s, resident);
    if (p[0].st.dup_found) throw std::runtime_error("a regrouped table is still not contiguous");
    settle(g, p);
}

// A scattered table, host text or device text, regrouped once -- on the GPU of the first context when regroup_gpu allows it,
// else on the host -- and run again for every configuration.  The regrouped text is ours: the results' strings are copied
// into pools.
void run_scattered(const Group& g, const char* h_text, const uint8_t* d_text, uint64_t n, cudaStream_t s) {
    blu_ctx* c = g[0].c;
    DevMem dt;
    if (regroup_gpu(c, h_text, d_text, n, s, dt)) {
        if (c->is_multi()) {
            // the shards start from host text: the regrouped table comes back once and is cut like any other
            std::string re((size_t)dt.n, '\0');
            CK(cudaMemcpy(re.data(), dt.p, dt.n, cudaMemcpyDeviceToHost));
            cudaFree(dt.p);
            dt.p = nullptr;
            run_table(g, ByteView(re.data(), re.size()), false);
        } else
            run_regrouped_device(g, dt, c->stream, false);
        c->tm.n_regrouped = 2;
        return;
    }
    std::string host;
    if (!h_text) {
        host.resize((size_t)n);
        CK(cudaMemcpy(host.data(), d_text, n, cudaMemcpyDeviceToHost));
        h_text = host.data();
    }
    const std::string re = regroup_by_query(h_text, n);
    std::string().swap(host);
    run_table(g, ByteView(re.data(), re.size()), false);
    c->tm.n_regrouped = 1;
}

std::unique_ptr<blu_result> new_result(blu_ctx* c) {
    auto r = std::make_unique<blu_result>();
    r->tax = c->is_multi() ? c->shards[0]->tax : c->tax;
    r->cut = c->cut;
    return r;
}

// the concatenation behind blu_result_records() & co. for a multi-part result
void merge_parts(const blu_result* r) {
    std::lock_guard<std::mutex> g(r->merge_mu);
    if (r->merged) return;
    uint64_t nr = 0, nb = 0, na = 0, np = 0;
    bool all_ext = true;
    const char* ext_lo = nullptr;
    const char* ext_hi = nullptr;
    for (auto& p : r->parts) {
        nr += p.n_rec, nb += p.n_beans, na += p.n_accs, np += p.strings_len();
        if (!p.n_rec) continue;
        if (!p.ext_strings) {
            all_ext = false;
            continue;
        }
        if (!ext_lo || p.ext_strings < ext_lo) ext_lo = p.ext_strings;
        if (!ext_hi || p.ext_strings + p.ext_len > ext_hi) ext_hi = p.ext_strings + p.ext_len;
    }
    all_ext = all_ext && ext_lo != nullptr;
    if (nb >= kIdxMax || na >= kIdxMax) throw UnsupportedErr("the concatenated result has more than 2^32 beans / accession references: read it part by part");
    r->m_rec.reserve(nr), r->m_beans.reserve(nb), r->m_accs.reserve(na);
    if (!all_ext) r->m_pool.reserve(np);
    for (auto& p : r->parts) {
        if (!p.n_rec) continue;
        // where this part's strings sit in the concatenation's string base
        const uint64_t b0 = r->m_beans.size(), a0 = r->m_accs.size(), s0 = all_ext ? (uint64_t)(p.ext_strings - ext_lo) : r->m_pool.size();
        const blu_record* rec = (const blu_record*)p.b_rec.p;
        for (uint64_t i = 0; i < p.n_rec; i++) {
            blu_record x = rec[i];
            x.bean_base += (uint32_t)b0, x.acc_base += (uint32_t)a0, x.query_off += s0;
            r->m_rec.push_back(x);
        }
        const blu_bean* bn = (const blu_bean*)p.b_beans.p;
        r->m_beans.insert(r->m_beans.end(), bn, bn + p.n_beans);
        const blu_acc* ac = (const blu_acc*)p.b_accs.p;
        for (uint64_t i = 0; i < p.n_accs; i++) r->m_accs.push_back(blu_acc{ac[i].ref + (s0 << 16)});
        if (!all_ext && p.strings_len()) r->m_pool.append(p.strings(), p.strings_len());
    }
    if (all_ext) r->m_ext = ext_lo, r->m_ext_len = (uint64_t)(ext_hi - ext_lo);
    r->merged = true;
}

// --- records in query-id order (blu_result_sort_by_query) ----------------------------------------------------------------
// BLU_SORT_TRACE=1: wall time of every stage on stderr (the stream is synchronised at each mark: measurement only)
struct SortTrace {
    bool on;
    cudaStream_t s;
    std::chrono::steady_clock::time_point t0;
    std::string line;
    explicit SortTrace(cudaStream_t st) : on(getenv("BLU_SORT_TRACE") != nullptr), s(st), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) {
        if (!on) return;
        cudaStreamSynchronize(s);
        const auto t1 = std::chrono::steady_clock::now();
        char b[96];
        snprintf(b, sizeof b, "%s%s %.3f", line.empty() ? "" : ", ", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        line += b;
        t0 = t1;
    }
    ~SortTrace() {
        if (on) fprintf(stderr, "[blu sort] ms: %s\n", line.c_str());
    }
};

// device scratch of one sort call
template <class T>
T* sort_scratch(DevMem& m, uint64_t count) {
    if (!m.alloc(std::max<uint64_t>(count, 1) * sizeof(T))) throw UnsupportedErr("the query ids and the sort's scratch do not fit the device");
    return (T*)m.p;
}

// the ids (id_bytes), their references, the permutation, `extra` bytes and the sort's scratch must fit the free device memory
void require_sort_fits(uint64_t n, uint64_t id_bytes, uint64_t extra) {
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t need = id_bytes + n * (sizeof(uint64_t) + 2 * sizeof(uint32_t)) + extra + sort_ids_device_bytes(n) + (64ull << 20);
    if (need > (uint64_t)free_b)
        throw UnsupportedErr("the query ids and the sort's scratch (" + std::to_string(need >> 20) + " MiB) do not fit the device (" +
                             std::to_string(free_b >> 20) + " MiB free)");
}

void sort_ids_checked(const uint8_t* base, const uint64_t* off, const uint32_t* len, uint32_t n, uint32_t* perm, cudaStream_t s) {
    const int rc = sort_ids_device(base, off, len, n, perm, s);
    if (rc == 1) throw UnsupportedErr("the sort's scratch does not fit the device");
    if (rc < 0) throw CudaErr(std::string("sort_ids_device: ") + cudaGetErrorString((cudaError_t)(-rc)));
}

// a device-resident part: the records are gathered in HBM into a record buffer of the context's DevicePool
void sort_part_device(blu_ctx* c, ResultPartOwned& p) {
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    const uint32_t n = (uint32_t)p.n_rec;
    SortTrace tr(s);
    require_sort_fits(n, 0, (uint64_t)n * sizeof(blu_record));
    DevMem m_off, m_len, m_perm;
    uint64_t* off = sort_scratch<uint64_t>(m_off, n);
    uint32_t* len = sort_scratch<uint32_t>(m_len, n);
    uint32_t* perm = sort_scratch<uint32_t>(m_perm, n);
    CK(launch_record_ids(p.dev->rec.p, n, off, len, s));
    sort_ids_checked(p.dtext, off, len, n, perm, s);
    tr.mark("sort");
    std::unique_ptr<DeviceSet> set = p.dev_pool->acquire();
    try {
        set->rec.ensure(n);
        CK(launch_gather_records(p.dev->rec.p, perm, n, set->rec.p, s));
        CK(cudaStreamSynchronize(s));
    } catch (...) {
        cudaStreamSynchronize(s);
        p.dev_pool->release(std::move(set));
        throw;
    }
    std::swap(p.dev->rec, set->rec);
    p.dev_pool->release(std::move(set));
    tr.mark("permute");
}

// the parts of a multi-device host result become one part (the concatenation merge_parts builds)
void concat_parts(blu_ctx* g, blu_result* r) {
    merge_parts(r);
    ResultPartOwned one;
    one.pinned = g->pool;
    try {
        auto put = [&](PinnedBuf& b, const void* src, uint64_t bytes) {
            b = g->acquire(std::max<uint64_t>(bytes, 64));
            if (bytes) memcpy(b.p, src, bytes);
        };
        put(one.b_rec, r->m_rec.data(), r->m_rec.size() * sizeof(blu_record));
        put(one.b_beans, r->m_beans.data(), r->m_beans.size() * sizeof(blu_bean));
        put(one.b_accs, r->m_accs.data(), r->m_accs.size() * sizeof(blu_acc));
        if (r->m_ext) {
            one.ext_strings = r->m_ext, one.ext_len = r->m_ext_len;
        } else {
            put(one.b_pool, r->m_pool.data(), r->m_pool.size());
            one.pool_len = r->m_pool.size();
        }
    } catch (...) {
        one.free_buffers();
        throw;
    }
    one.n_rec = r->m_rec.size(), one.n_beans = r->m_beans.size(), one.n_accs = r->m_accs.size();
    for (auto& p : r->parts) p.free_buffers();
    r->parts.clear();
    r->parts.push_back(std::move(one));
    std::lock_guard<std::mutex> lk(r->merge_mu);
    r->merged = false;
    std::vector<blu_record>().swap(r->m_rec);
    std::vector<blu_bean>().swap(r->m_beans);
    std::vector<blu_acc>().swap(r->m_accs);
    std::string().swap(r->m_pool);
    r->m_ext = nullptr, r->m_ext_len = 0;
}

// a host part: its ids are packed into pinned memory and sorted on g's GPU; the permutation comes back and the records are
// gathered on all host threads
void sort_part_host(blu_ctx* g, ResultPartOwned& p) {
    const uint64_t n = p.n_rec;
    const blu_record* rec = (const blu_record*)p.b_rec.p;
    const char* str = p.strings();
    cudaStream_t s = g->stream;
    struct Pinned {
        std::shared_ptr<PinnedPool> pool;
        PinnedBuf b;
        ~Pinned() { pool->release(b); }
    };
    SortTrace tr(s);
    Pinned h_off{g->pool, g->acquire(n * sizeof(uint64_t))}, h_len{g->pool, g->acquire(n * sizeof(uint32_t))};
    uint64_t* off = (uint64_t*)h_off.b.p;
    uint32_t* len = (uint32_t*)h_len.b.p;
    std::vector<uint64_t> sums(host_threads() + 1, 0);
    parallel_ranges(n, [&](unsigned t, size_t a, size_t b) {
        uint64_t x = 0;
        for (size_t i = a; i < b; i++) x += rec[i].query_len;
        sums[t + 1] = x;
    });
    for (size_t t = 1; t < sums.size(); t++) sums[t] += sums[t - 1];
    const uint64_t id_bytes = sums.back();
    Pinned h_ids{g->pool, g->acquire(std::max<uint64_t>(id_bytes, 64))};
    char* ids = (char*)h_ids.b.p;
    parallel_ranges(n, [&](unsigned t, size_t a, size_t b) {
        uint64_t o = sums[t];
        for (size_t i = a; i < b; i++) {
            off[i] = o, len[i] = rec[i].query_len;
            memcpy(ids + o, str + rec[i].query_off, rec[i].query_len);
            o += rec[i].query_len;
        }
    });
    tr.mark("pack");
    require_sort_fits(n, id_bytes, 0);
    Pinned h_perm{g->pool, g->acquire(n * sizeof(uint32_t))};
    {
        DevMem m_ids, m_off, m_len, m_perm;
        uint8_t* d_ids = sort_scratch<uint8_t>(m_ids, id_bytes);
        uint64_t* d_off = sort_scratch<uint64_t>(m_off, n);
        uint32_t* d_len = sort_scratch<uint32_t>(m_len, n);
        uint32_t* d_perm = sort_scratch<uint32_t>(m_perm, n);
        try {
            if (id_bytes) CK(cudaMemcpyAsync(d_ids, ids, id_bytes, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(d_off, off, n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(d_len, len, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
            tr.mark("h2d");
            sort_ids_checked(d_ids, d_off, d_len, (uint32_t)n, d_perm, s);
            tr.mark("sort");
            CK(cudaMemcpyAsync(h_perm.b.p, d_perm, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            tr.mark("d2h");
        } catch (...) {  // nothing may still be copying when the buffers go back to their pools
            cudaStreamSynchronize(s);
            throw;
        }
    }
    const uint32_t* perm = (const uint32_t*)h_perm.b.p;
    PinnedBuf out = p.pinned->acquire(n * sizeof(blu_record));
    blu_record* dst = (blu_record*)out.p;
    parallel_ranges(n, [&](unsigned, size_t a, size_t b) {
        for (size_t i = a; i < b; i++) dst[i] = rec[perm[i]];
    });
    p.pinned->release(p.b_rec);
    p.b_rec = out;
    tr.mark("permute");
}

// A pass with several configurations: every context reports the shared pass -- the first one's launches, copies and kernel
// times -- and the bytes all of them downloaded; result and taxonomy bytes stay each context's own.
void share_timings(const std::vector<blu_ctx*>& cs) {
    if (cs.size() < 2) return;
    uint64_t d2h = 0;
    for (blu_ctx* c : cs) d2h += c->tm.d2h_bytes;
    for (blu_ctx* c : cs) {
        const uint64_t result = c->tm.result_bytes, tax = c->tm.taxonomy_bytes;
        c->tm = cs[0]->tm;
        c->tm.result_bytes = result, c->tm.taxonomy_bytes = tax, c->tm.d2h_bytes = d2h;
    }
}

// What every blu_consensus_run_* entry point does with its results: one per context, made for `run`, handed out on
// success, all freed on failure; the message of a failure goes to every context.
template <class F>
int run_entry(const std::vector<blu_ctx*>& cs, blu_result** outs, F&& run) {
    std::vector<std::unique_ptr<blu_result>> rs;
    const int rc = guarded(cs[0], [&] {
        Group g;
        for (blu_ctx* c : cs) {
            require_tax(c);
            rs.push_back(new_result(c));
            g.push_back(Member{c, rs.back().get()});
        }
        run(g);
        share_timings(cs);
    });
    for (blu_ctx* c : cs) c->err = cs[0]->err;
    if (rc != BLU_OK) {
        for (auto& r : rs) blu_result_free(r.release());
        return rc;
    }
    for (size_t i = 0; i < rs.size(); i++) outs[i] = rs[i].release();
    return BLU_OK;
}

int fail_all(const std::vector<blu_ctx*>& cs, int code, const std::string& msg) {
    for (blu_ctx* c : cs) fail(c, code, msg);
    return code;
}

// blu_consensus_run_host and _host_configs
int host_entry(const std::vector<blu_ctx*>& cs, const char* text, uint64_t n, blu_result** outs) {
    return run_entry(cs, outs, [&](const Group& g) {
        try {
            run_table(g, ByteView(text, n), (g[0].c->opts.flags & BLU_OPT_TEXT_REFS) != 0);
        } catch (const NonContiguous&) {
            run_scattered(g, text, nullptr, n, g[0].c->stream);
        }
    });
}

// blu_consensus_run_file and _file_configs: the file is streamed (FileSource); only a non-contiguous table (regrouping needs
// all rows at once) is read whole.
int file_entry(const std::vector<blu_ctx*>& cs, const char* path, blu_result** outs) {
    struct Fd {
        int fd;
        ~Fd() {
            if (fd >= 0) close(fd);
        }
    } f{open(path, O_RDONLY | O_CLOEXEC)};
    struct stat st;
    if (f.fd < 0 || fstat(f.fd, &st) != 0 || !S_ISREG(st.st_mode))
        return fail_all(cs, BLU_ERR_IO, "Unexpected error occurred on load table.");  // mod.rs:357-364
    const uint64_t n = (uint64_t)st.st_size;
    return run_entry(cs, outs, [&](const Group& g) {
        if (n == 0) throw DataErr("empty blast output (the reference's CsvReader fails on an empty file)");
        try {
            run_table(g, ByteView(f.fd, n), false);
        } catch (const NonContiguous&) {
            std::string all((size_t)n, '\0');
            for (uint64_t off = 0; off < n;) {
                ssize_t got = pread(f.fd, all.data() + off, (size_t)std::min<uint64_t>(n - off, 1ull << 30), (off_t)off);
                if (got < 0 && errno == EINTR) continue;
                if (got <= 0) throw IoErr("Unexpected error occurred on load table.");
                off += (uint64_t)got;
            }
            run_scattered(g, all.data(), nullptr, n, g[0].c->stream);
        }
    });
}

// blu_consensus_run_device_resident and _device_resident_configs
int resident_entry(const std::vector<blu_ctx*>& cs, const void* dtext, uint64_t n, void* stream, blu_result** outs) {
    return run_entry(cs, outs, [&](const Group& g) {
        blu_ctx* c = g[0].c;
        CK(cudaSetDevice(c->device));
        cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
        Pass p = new_pass(g);
        run_device_text(p, (const uint8_t*)dtext, n, s, true);
        if (!p[0].st.dup_found) {
            settle(g, p);
            return;
        }
        // a scattered table: regrouped in HBM (blu_regroup.cu); the results' references then point into that copy, which
        // the results own together (blu_result_device_text)
        DevMem dt;
        if (!regroup_gpu(c, nullptr, (const uint8_t*)dtext, n, s, dt))
            throw UnsupportedErr("the table's queries are not contiguous and it cannot be regrouped on the device: use blu_consensus_run_device / _host / _file");
        run_regrouped_device(g, dt, s, true);
        const std::shared_ptr<uint8_t> owned(dt.p, [](uint8_t* q) { cudaFree(q); });
        dt.p = nullptr;
        for (const Member& m : g) m.r->parts[0].owned_dtext = owned;
        c->tm.n_regrouped = 2;
    });
}

// The rules of a group of configurations (include/blu_consensus.h); the message of the first one broken, or "".
std::string group_error(const std::vector<blu_ctx*>& cs) {
    const blu_ctx* c0 = cs[0];
    for (size_t i = 0; i < cs.size(); i++) {
        const blu_ctx* c = cs[i];
        const std::string at = "ctxs[" + std::to_string(i) + "]: ";
        if (c->is_multi()) return at + "a multi-device context cannot be part of a group of configurations";
        if (!c->tax) return at + "no taxonomy loaded (call blu_taxonomy_load_json first)";
        for (size_t j = 0; j < i; j++)
            if (cs[j] == c) return at + "the same context as ctxs[" + std::to_string(j) + "]";
        if (c->device != c0->device) return at + "on another device than ctxs[0]";
        if (c->opts.chunk_bytes != c0->opts.chunk_bytes) return at + "chunk_bytes differs from that of ctxs[0]";
        if (c->opts.flags != c0->opts.flags) return at + "flags differ from those of ctxs[0]";
    }
    return "";
}

// Checks the arguments every _configs entry point takes: 0 and the contexts in `cs`, or the error code.  The message goes to
// every context listed and to blu_last_error(NULL).
int take_group(blu_ctx* const* ctxs, int n, blu_result** outs, std::vector<blu_ctx*>& cs) {
    auto refuse = [&](const std::string& msg) {
        fail(nullptr, BLU_ERR_ARG, msg);
        for (int i = 0; ctxs && i < n; i++)
            if (ctxs[i]) fail(ctxs[i], BLU_ERR_ARG, msg);
        return BLU_ERR_ARG;
    };
    if (!ctxs || n < 1 || n > kMaxConfigs) return refuse("a group holds 1 to 8 contexts");
    for (int i = 0; i < n; i++)
        if (!ctxs[i]) return refuse("ctxs[" + std::to_string(i) + "] is null");
    if (!outs) return refuse("null argument");
    cs.assign(ctxs, ctxs + n);
    for (int i = 0; i < n; i++) outs[i] = nullptr;
    if (n == 1) return BLU_OK;
    const std::string e = group_error(cs);
    return e.empty() ? BLU_OK : refuse(e);
}

}  // namespace

// =================================================================================================================
// C ABI
// =================================================================================================================
extern "C" {

int blu_abi_version(void) { return BLU_ABI_VERSION; }

const char* blu_last_error(const blu_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

static int validate_opts(const blu_opts* opts) {
    if (opts->taxon < 0 || opts->taxon > 3) return fail(nullptr, BLU_ERR_ARG, "bad taxon");
    if (opts->strategy < 0 || opts->strategy > 1) return fail(nullptr, BLU_ERR_ARG, "bad strategy");
    if (opts->taxon == BLU_TAXON_CUSTOM && !opts->has_custom)
        return fail(nullptr, BLU_ERR_DATA, "Custom taxon values are required when the custom taxon option is selected.");
    return BLU_OK;
}

static void fill_cutoffs(blu_ctx* c, const blu_opts* opts) {
    c->opts = *opts;
    c->cut.taxon = opts->taxon;
    c->cut.has_custom = opts->has_custom != 0;
    for (int i = 0; i < 8; i++) c->cut.custom[i] = opts->custom[i];
}

int blu_ctx_create(const blu_opts* opts, blu_ctx** out) {
    if (!opts || !out) return fail(nullptr, BLU_ERR_ARG, "null argument");
    *out = nullptr;
    if (int rc = validate_opts(opts)) return rc;
    auto c = std::make_unique<blu_ctx>();
    fill_cutoffs(c.get(), opts);
    c->device = opts->device;
    c->dev_pool->device = opts->device;
    int rc = guarded(nullptr, [&] {
        make_backbone(c->cut);  // validates the custom values
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0) throw CudaErr(std::string("no CUDA device available: ") + cudaGetErrorString(e));
        if (c->device < 0 || c->device >= n) throw CudaErr("device ordinal out of range");
        CK(cudaSetDevice(c->device));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, c->device));
        if (prop.major < 10) throw CudaErr(std::string("device '") + prop.name + "' is not sm_100-class; this library only carries sm_100a code");
        c->sms = prop.multiProcessorCount;
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
        for (auto& row : c->ev)
            for (auto& e2 : row) CK(cudaEventCreate(&e2));
        for (auto& e2 : c->ev_h2d) CK(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        for (auto& e2 : c->ev_free) CK(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        CK(cudaMalloc((void**)&c->d_ctr, sizeof(Counters)));
        // counter snapshots: written by advance_kernel straight into (mapped) host memory
        CK(cudaHostAlloc((void**)&c->h_snap, kMaxRanges * sizeof(Counters), cudaHostAllocMapped | cudaHostAllocPortable));
        CK(cudaHostGetDevicePointer((void**)&c->d_snap, c->h_snap, 0));
        CK(kernels_set_attributes());
    });
    if (rc != BLU_OK) {
        std::string msg = g_create_error;
        blu_ctx_destroy(c.release());
        g_create_error = msg;
        return rc;
    }
    *out = c.release();
    return BLU_OK;
}

int blu_ctx_create_multi(const blu_opts* opts, const int* devices, int n_devices, blu_ctx** out) {
    if (!opts || !out || !devices || n_devices < 1 || n_devices > 64) return fail(nullptr, BLU_ERR_ARG, "bad argument");
    *out = nullptr;
    if (int rc = validate_opts(opts)) return rc;
    for (int i = 0; i < n_devices; i++)
        for (int j = 0; j < i; j++)
            if (devices[i] == devices[j]) return fail(nullptr, BLU_ERR_ARG, "a device is listed twice");
    auto c = std::make_unique<blu_ctx>();
    fill_cutoffs(c.get(), opts);
    c->device = devices[0];
    for (int i = 0; i < n_devices; i++) {
        blu_opts o = *opts;
        o.device = devices[i];
        blu_ctx* sh = nullptr;
        int rc = blu_ctx_create(&o, &sh);
        if (rc != BLU_OK) {
            std::string msg = g_create_error;
            blu_ctx_destroy(c.release());
            g_create_error = msg;
            return rc;
        }
        sh->keep_hashes = true;
        c->shards.emplace_back(sh);
    }
    *out = c.release();
    return BLU_OK;
}

int blu_ctx_num_devices(const blu_ctx* c) { return !c ? 0 : (c->is_multi() ? (int)c->shards.size() : 1); }

void blu_ctx_destroy(blu_ctx* c) {
    if (!c) return;
    if (c->is_multi()) {
        for (auto& sh : c->shards) blu_ctx_destroy(sh.release());
        delete c;
        return;
    }
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->d2h_stream) cudaStreamSynchronize(c->d2h_stream);
    c->d_lin_off.release(), c->d_lvl.release(), c->d_bean.release(), c->d_irank.release(), c->d_cut.release();
    c->d_rcls.release(), c->d_acls.release(), c->d_linok.release(), c->d_slots.release();
    c->d_text[0].release(), c->d_text[1].release();
    if (c->out) c->out->release();
    c->dev_pool->close();
    c->d_defer.release(), c->d_pool.release(), c->d_dup.release(), c->d_top.release(), c->d_qhash.release();
    c->d_big_rows.release(), c->d_big_cand.release();
    if (c->d_ctr) cudaFree(c->d_ctr);
    if (c->h_snap) cudaFreeHost(c->h_snap);
    c->pool->close();
    for (auto& row : c->ev)
        for (auto& e : row)
            if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_h2d)
        if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_free)
        if (e) cudaEventDestroy(e);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    delete c;
}

int blu_custom_cutoffs_from_file(const char* path, blu_opts* opts, char* err, size_t errlen) {
    if (!path || !opts) return BLU_ERR_ARG;
    try {
        Cutoffs c;
        read_custom_cutoffs(path, c);
        opts->has_custom = 1;
        for (int i = 0; i < 8; i++) opts->custom[i] = c.custom[i];
        return BLU_OK;
    } catch (const std::exception& e) {
        if (err && errlen) snprintf(err, errlen, "%s", e.what());
        return BLU_ERR_DATA;  // the reference panics on every failure of CustomTaxon::from_file
    }
}

// the encoded lineage tables go to every GPU of the context (replicated: SURVEY 8e)
static void install_taxonomy(blu_ctx* c, const std::shared_ptr<HostTaxonomy>& T) {
    if (!c->is_multi()) {
        CK(cudaSetDevice(c->device));
        c->tax = T;
        upload_taxonomy(c);
        c->dens_rec = 0;  // (a different taxonomy usually comes with a different kind of table)
        return;
    }
    c->tax = T;
    for (auto& sh : c->shards) install_taxonomy(sh.get(), T);
}

int blu_taxonomy_load_arrays(blu_ctx* c, const int64_t* taxids, const uint64_t* off, const char* blob, uint64_t n) {
    if (!c || (n && (!taxids || !off || !blob))) return fail(c, BLU_ERR_ARG, "null argument");
    return guarded(c, [&] {
        auto T = std::make_shared<HostTaxonomy>();
        static const uint64_t zero = 0;
        build_taxonomy(taxids, n ? off : &zero, blob, n, c->cut, *T);
        install_taxonomy(c, T);
    });
}

int blu_taxonomy_load_json(blu_ctx* c, const char* path) {
    if (!c || !path) return fail(c, BLU_ERR_ARG, "null argument");
    std::vector<int64_t> ids;
    std::vector<uint64_t> off;
    std::string blob;
    int rc = guarded(c, [&] { read_taxonomy_json(path, c->opts.use_taxid != 0, ids, off, blob); });
    if (rc != BLU_OK) return rc;
    return blu_taxonomy_load_arrays(c, ids.data(), off.data(), blob.data(), ids.size());
}

int blu_taxonomy_load_json_cached(blu_ctx* c, const char* path, const char* cache_path, int* cache_state) {
    if (!c || !path) return fail(c, BLU_ERR_ARG, "null argument");
    if (cache_state) *cache_state = 0;
    const std::string cpath = cache_path ? std::string(cache_path) : std::string(path) + ".blucache";
    return guarded(c, [&] {
        const TaxCacheKey key = make_cache_key(path, c->opts.use_taxid != 0, c->cut);  // IoErr if the JSON is unreadable
        auto T = std::make_shared<HostTaxonomy>();
        int state = 1;
        if (!load_taxonomy_cache(cpath.c_str(), key, *T)) {
            std::vector<int64_t> ids;
            std::vector<uint64_t> off;
            std::string blob;
            read_taxonomy_json(path, c->opts.use_taxid != 0, ids, off, blob);
            static const uint64_t zero = 0;
            build_taxonomy(ids.data(), ids.empty() ? &zero : off.data(), blob.data(), ids.size(), c->cut, *T);
            state = 0;
            try {
                save_taxonomy_cache(cpath.c_str(), key, *T);
            } catch (const IoErr&) {
                state = -1;
            }
        }
        install_taxonomy(c, T);
        if (cache_state) *cache_state = state;
    });
}

int blu_consensus_run_device(blu_ctx* c, const void* dtext, uint64_t n, void* stream, blu_result** out) {
    if (!c || !out || (!dtext && n)) return fail(c, BLU_ERR_ARG, "null argument");
    *out = nullptr;
    if (c->is_multi()) return fail(c, BLU_ERR_ARG, "device-resident text belongs to one GPU: use a single-device context");
    return run_entry({c}, out, [&](const Group& g) {
        CK(cudaSetDevice(c->device));
        cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
        try {
            Pass p = new_pass(g);
            run_device_text(p, (const uint8_t*)dtext, n, s, false);
            settle(g, p);
        } catch (const NonContiguous&) {
            run_scattered(g, nullptr, (const uint8_t*)dtext, n, s);
        }
    });
}

int blu_consensus_run_device_resident(blu_ctx* c, const void* dtext, uint64_t n, void* stream, blu_result** out) {
    if (!c || !out || (!dtext && n)) return fail(c, BLU_ERR_ARG, "null argument");
    *out = nullptr;
    if (c->is_multi()) return fail(c, BLU_ERR_ARG, "device-resident text belongs to one GPU: use a single-device context");
    return resident_entry({c}, dtext, n, stream, out);
}

int blu_consensus_run_device_resident_configs(blu_ctx* const* ctxs, int n_ctx, const void* dtext, uint64_t n, void* stream, blu_result** outs) {
    std::vector<blu_ctx*> cs;
    if (int rc = take_group(ctxs, n_ctx, outs, cs)) return rc;
    if (n_ctx == 1) return blu_consensus_run_device_resident(cs[0], dtext, n, stream, outs);
    if (!dtext && n) return fail_all(cs, BLU_ERR_ARG, "null argument");
    return resident_entry(cs, dtext, n, stream, outs);
}

const void* blu_result_device_text(const blu_result* r, uint64_t* n) {
    const bool ok = r && r->parts.size() == 1 && r->parts[0].dev;
    if (n) *n = ok ? r->parts[0].dtext_len : 0;
    return ok ? r->parts[0].dtext : nullptr;
}
const blu_record* blu_result_device_records(const blu_result* r) {
    return (r && r->parts.size() == 1 && r->parts[0].dev) ? r->parts[0].dev->rec.p : nullptr;
}
const blu_bean* blu_result_device_beans(const blu_result* r, uint64_t* n) {
    const bool ok = r && r->parts.size() == 1 && r->parts[0].dev;
    if (n) *n = ok ? r->parts[0].n_beans : 0;
    return ok ? r->parts[0].dev->beans.p : nullptr;
}
const blu_acc* blu_result_device_accessions(const blu_result* r, uint64_t* n) {
    const bool ok = r && r->parts.size() == 1 && r->parts[0].dev;
    if (n) *n = ok ? r->parts[0].n_accs : 0;
    return ok ? r->parts[0].dev->accs.p : nullptr;
}

int blu_result_download(blu_result* r) {
    if (!r) return BLU_ERR_ARG;
    try {
        for (auto& p : r->parts) download_part(&p);
        return BLU_OK;
    } catch (const CudaErr&) {
        return BLU_ERR_CUDA;
    } catch (const std::exception&) {
        return BLU_ERR_INTERNAL;
    }
}

int blu_result_sort_by_query(blu_ctx* c, blu_result* r) {
    if (!c || !r) return fail(c, BLU_ERR_ARG, "null argument");
    if (!r->on_host() && (r->parts.size() != 1 || r->parts[0].ctx != c))
        return fail(c, BLU_ERR_ARG, "a device-resident result is sorted with the context that produced it");
    return guarded(c, [&] {
        const uint64_t n = r->n_rec();
        if (n == 0) return;
        if (n > 0xFFFFFFFFull) throw UnsupportedErr("more than 2^32 - 1 records");
        if (!r->on_host()) {
            sort_part_device(c, r->parts[0]);
        } else {
            blu_ctx* g = c->is_multi() ? c->shards[0].get() : c;
            CK(cudaSetDevice(g->device));
            if (r->parts.size() > 1) concat_parts(g, r);
            sort_part_host(g, r->parts[0]);
        }
        r->sorted = true;
    });
}

int blu_consensus_run_host(blu_ctx* c, const char* text, uint64_t n, blu_result** out) {
    if (!c || !out || (!text && n)) return fail(c, BLU_ERR_ARG, "null argument");
    *out = nullptr;
    return host_entry({c}, text, n, out);
}

int blu_consensus_run_host_configs(blu_ctx* const* ctxs, int n_ctx, const char* text, uint64_t n, blu_result** outs) {
    std::vector<blu_ctx*> cs;
    if (int rc = take_group(ctxs, n_ctx, outs, cs)) return rc;
    if (n_ctx == 1) return blu_consensus_run_host(cs[0], text, n, outs);
    if (!text && n) return fail_all(cs, BLU_ERR_ARG, "null argument");
    return host_entry(cs, text, n, outs);
}

int blu_consensus_run_file(blu_ctx* c, const char* path, blu_result** out) {
    if (!c || !path || !out) return fail(c, BLU_ERR_ARG, "null argument");
    *out = nullptr;
    return file_entry({c}, path, out);
}

int blu_consensus_run_file_configs(blu_ctx* const* ctxs, int n_ctx, const char* path, blu_result** outs) {
    std::vector<blu_ctx*> cs;
    if (int rc = take_group(ctxs, n_ctx, outs, cs)) return rc;
    if (n_ctx == 1) return blu_consensus_run_file(cs[0], path, outs);
    if (!path) return fail_all(cs, BLU_ERR_ARG, "null argument");
    return file_entry(cs, path, outs);
}

int blu_result_add_headers(blu_result* r, const char* headers_nl, uint64_t len) {
    if (!r || !r->on_host()) return BLU_ERR_ARG;
    std::unordered_set<std::string_view> have;
    have.reserve(r->n_rec() * 2);
    for (auto& p : r->parts) {
        const blu_record* rec = (const blu_record*)p.b_rec.p;
        for (uint64_t i = 0; i < p.n_rec; i++) have.insert(std::string_view(p.strings() + rec[i].query_off, rec[i].query_len));
    }
    const char* p = headers_nl;
    const char* e = headers_nl + len;
    while (p < e) {
        const char* nl = (const char*)memchr(p, '\n', e - p);
        const char* le = nl ? nl : e;
        std::string_view h(p, le - p);
        if (!have.count(h)) r->hitless.emplace_back(h);  // duplicates in `headers` stay duplicated, as in the reference
        p = le + 1;
    }
    return BLU_OK;
}

uint64_t blu_result_num_queries(const blu_result* r) { return r ? r->n_rec() + r->hitless.size() : 0; }
uint64_t blu_result_num_records(const blu_result* r) { return r ? r->n_rec() : 0; }
uint64_t blu_result_num_rows(const blu_result* r) { return r ? r->n_rows : 0; }
uint64_t blu_result_num_beans(const blu_result* r) {
    uint64_t n = 0;
    if (r)
        for (auto& p : r->parts) n += p.n_beans;
    return n;
}
uint64_t blu_result_num_accessions(const blu_result* r) {
    uint64_t n = 0;
    if (r)
        for (auto& p : r->parts) n += p.n_accs;
    return n;
}

static bool host_arrays(const blu_result* r) {
    if (!r || !r->on_host() || r->parts.empty()) return false;
    if (r->parts.size() > 1) {
        try {
            merge_parts(r);
        } catch (const std::exception&) {
            return false;
        }
    }
    return true;
}
const blu_record* blu_result_records(const blu_result* r) {
    if (!host_arrays(r)) return nullptr;
    return r->parts.size() == 1 ? (const blu_record*)r->parts[0].b_rec.p : r->m_rec.data();
}
const blu_bean* blu_result_beans(const blu_result* r) {
    if (!host_arrays(r)) return nullptr;
    return r->parts.size() == 1 ? (const blu_bean*)r->parts[0].b_beans.p : r->m_beans.data();
}
const blu_acc* blu_result_accessions(const blu_result* r) {
    if (!host_arrays(r)) return nullptr;
    return r->parts.size() == 1 ? (const blu_acc*)r->parts[0].b_accs.p : r->m_accs.data();
}
const char* blu_result_pool(const blu_result* r, uint64_t* len) {
    if (len) *len = 0;
    if (!host_arrays(r)) return nullptr;
    if (r->parts.size() == 1) {
        if (len) *len = r->parts[0].strings_len();
        return r->parts[0].strings();
    }
    if (r->m_ext) {
        if (len) *len = r->m_ext_len;
        return r->m_ext;
    }
    if (len) *len = r->m_pool.size();
    return r->m_pool.data();
}

uint64_t blu_result_checksum(const blu_result* r) {
    if (!r || !r->on_host()) return 0;
    ResultView v = make_view(r);
    return view_checksum(&v);
}

int blu_result_to_jsonl_head(const blu_result* r, uint64_t max_entries, char** out, uint64_t* len) {
    if (!r || !out || !len || !r->on_host()) return BLU_ERR_ARG;
    try {
        ResultView v = make_view(r);
        std::string s = view_to_jsonl(&v, max_entries);
        char* buf = (char*)malloc(s.size() + 1);
        if (!buf) return BLU_ERR_INTERNAL;
        memcpy(buf, s.data(), s.size());
        buf[s.size()] = 0;
        *out = buf;
        *len = s.size();
        return BLU_OK;
    } catch (const std::exception&) {
        return BLU_ERR_INTERNAL;
    }
}

int blu_result_to_jsonl(const blu_result* r, char** out, uint64_t* len) { return blu_result_to_jsonl_head(r, ~0ull, out, len); }

int blu_result_write(const blu_result* r, const char* path, int format, const char* run_id_in) {
    if (!r || format < 0 || format > 2 || !r->on_host()) return BLU_ERR_ARG;
    try {
        ResultView v = make_view(r);
        return view_write(&v, path, format, run_id_in);
    } catch (const std::exception&) {
        return BLU_ERR_INTERNAL;
    }
}

int blu_result_write_tabular(const blu_result* r, const char* path, const char* run_id) {
    if (!r || !r->on_host()) return BLU_ERR_ARG;
    try {
        ResultView v = make_view(r);
        return view_write_tabular(&v, path, run_id);
    } catch (const std::exception&) {
        return BLU_ERR_INTERNAL;
    }
}

int blu_result_file_to_tabular(const char* in_path, const char* out_path, int input_format, const char* run_id, char* err, size_t errlen) {
    std::string msg;
    int rc;
    try {
        rc = result_file_to_tabular(in_path, out_path, input_format, run_id, msg);
    } catch (const std::exception& e) {
        msg = e.what();
        rc = BLU_ERR_INTERNAL;
    }
    if (rc != BLU_OK && err && errlen) snprintf(err, errlen, "%s", msg.c_str());
    return rc;
}

void blu_result_free(blu_result* r) {
    if (!r) return;
    for (auto& p : r->parts) p.free_buffers();
    delete r;
}

void blu_free(void* p) { free(p); }

int blu_ctx_last_timings(const blu_ctx* c, blu_timings* out) {
    if (!c || !out) return BLU_ERR_ARG;
    *out = c->tm;
    return BLU_OK;
}

static int measure_copy(blu_ctx* c, uint64_t bytes, double* gbps, bool to_device) {
    if (!c || !gbps || !bytes) return BLU_ERR_ARG;
    if (c->is_multi()) c = c->shards[0].get();
    return guarded(c, [&] {
        CK(cudaSetDevice(c->device));
        void* h = nullptr;
        void* d = nullptr;
        CK(cudaHostAlloc(&h, bytes, cudaHostAllocDefault));
        if (cudaMalloc(&d, bytes) != cudaSuccess) {
            cudaFreeHost(h);
            throw CudaErr("cudaMalloc failed");
        }
        memset(h, 1, bytes);
        // sustained, not best-of: one warm-up copy, then enough back-to-back copies for ~6 GB, timed as a whole -- on a box where
        // several GPUs copy at once a best-of figure picks the moments the others pause
        auto copy = [&] {
            if (to_device)
                cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c->stream);
            else
                cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, c->stream);
        };
        copy();
        cudaStreamSynchronize(c->stream);
        const int reps = (int)std::max<uint64_t>(2, (6ull << 30) / bytes);
        cudaEventRecord(c->ev[0][0], c->stream);
        for (int i = 0; i < reps; i++) copy();
        cudaEventRecord(c->ev[0][1], c->stream);
        cudaStreamSynchronize(c->stream);
        const double ms = ev_ms(c->ev[0][0], c->ev[0][1]);
        const double best = ms > 0 ? (double)bytes * reps / ms / 1e6 : 0;
        cudaFree(d);
        cudaFreeHost(h);
        *gbps = best;
    });
}
int blu_ctx_measure_h2d(blu_ctx* c, uint64_t bytes, double* gbps) { return measure_copy(c, bytes, gbps, true); }
int blu_ctx_measure_d2h(blu_ctx* c, uint64_t bytes, double* gbps) { return measure_copy(c, bytes, gbps, false); }

int blu_shard_cuts(const char* text, uint64_t n, int n_shards, uint64_t* cuts) {
    if (!cuts || n_shards < 1 || (!text && n)) return BLU_ERR_ARG;
    shard_cuts(ByteView(text, n), n_shards, cuts);
    return BLU_OK;
}

int blu_shard_cuts_file(const char* path, int n_shards, uint64_t* cuts) {
    if (!path || !cuts || n_shards < 1) return BLU_ERR_ARG;
    const int fd = open(path, O_RDONLY | O_CLOEXEC);
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) {
        if (fd >= 0) close(fd);
        return BLU_ERR_IO;
    }
    int rc = BLU_OK;
    try {
        shard_cuts(ByteView(fd, (uint64_t)st.st_size), n_shards, cuts);
    } catch (const std::exception&) {
        rc = BLU_ERR_IO;
    }
    close(fd);
    return rc;
}

void* blu_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;  // (portable: every GPU of a multi-device context copies from it)
    return p;
}
void blu_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

}  // extern "C"
