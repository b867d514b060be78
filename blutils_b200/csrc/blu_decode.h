// blu_decode.h -- host-side decoding of the binary consensus records into the reference's result objects and
// the writer of `write_blutils_output` (reference core/src/use_cases/write_blutils_output.rs:33-250), and the TSV layout of
// build-tabular that blu_tabular.h shares.
// Header-only so that the C ABI (blu_api.cpp) and the test-only host simulation (tests/csrc) share it.
#pragma once
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <cstdio>
#include <memory>
#include <cstring>
#include <filesystem>
#include <random>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "../../include/blu_consensus.h"
#include "blu_json.h"
#include "blu_taxonomy.h"

namespace blu {

// One part of a result set: the records one GPU produced, with the arrays their indices refer to.
struct ResultPart {
    const blu_record* rec = nullptr;
    const blu_bean* beans = nullptr;
    const blu_acc* accs = nullptr;
    const char* pool = nullptr;  // string base of this part: its string pool, or the text the references point into
    uint64_t n_rec = 0;
};

// Non-owning view of one result set (a multi-device run has one part per GPU; nothing is concatenated to decode it).
struct ResultView {
    const HostTaxonomy* tax = nullptr;
    Cutoffs cut;
    std::vector<ResultPart> parts;
    const std::vector<std::string>* hitless_ = nullptr;
    bool sorted = false;  // the records of the parts, in part order, are in query-id order already
    uint64_t n_rec() const {
        uint64_t n = 0;
        for (auto& p : parts) n += p.n_rec;
        return n;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// decoding: records -> the reference's result objects
// ---------------------------------------------------------------------------------------------------------------
inline std::string_view rec_query(const ResultPart& p, const blu_record& rc) { return std::string_view(p.pool + rc.query_off, rc.query_len); }

// serde_yaml 0.9 scalars (defined below)
inline void yaml_str(std::string& o, std::string_view s);
inline void yaml_f64(std::string& o, double v);

// A field is built here before it is escaped or placed: one string per thread, so no allocation per record.
inline std::string& scratch() {
    thread_local std::string s;
    s.clear();
    return s;
}

struct Decoder {
    const HostTaxonomy& T;
    std::vector<uint8_t> in_bb;  // per rank id: default rank present in the cutoff backbone
    explicit Decoder(const ResultView* r) : T(*r->tax) {
        auto bb = make_backbone(r->cut);
        in_bb.resize(T.ranks.size());
        for (size_t i = 0; i < T.ranks.size(); i++) {
            in_bb[i] = 0;
            if (T.ranks[i].def >= 0)
                for (auto& b : bb)
                    if (b.def == T.ranks[i].def) in_bb[i] = 1;
        }
    }

    // ---- the fields of a record: the writers read the taxonomy tables through these only ----
    // TaxonomyBean (taxonomy_bean.rs:5-17)
    std::string_view reached_rank(const blu_record& rc) const { return T.ranks[T.pos_rank[T.lin_off[rc.ref_lineage] + rc.reached_pos]].full; }
    // serde form of Option<LinnaeanRank> for max_allowed_rank (bbci.rs:22-30), nullptr = None: DefaultRank -> the enum variant,
    // NonDefaultRank(name) -> Other(name) where name = rank.to_string()
    const std::string* allowed_rank(const blu_record& rc) const {
        if (rc.allowed_pos < 0) return nullptr;
        const uint32_t k = T.pos_rank[T.lin_off[rc.ref_lineage] + rc.allowed_pos];
        return in_bb[k] ? &T.ranks[k].full : &T.ranks[k].display;
    }
    std::string_view identifier(const blu_record& rc) const { return T.idents[T.pos_ident[T.lin_off[rc.ref_lineage] + rc.reached_pos]]; }
    // `taxonomy`: the kept positions of the reference lineage
    void append_taxonomy(std::string& o, const blu_record& rc) const {
        const uint32_t lo = T.lin_off[rc.ref_lineage];
        bool first = true;
        for (int j = 0; j < T.lin_len(rc.ref_lineage); j++)
            if (rc.keep_mask >> j & 1) {
                if (!first) o.push_back(';');
                first = false;
                T.append_bean(o, lo + j);
            }
    }
    // ConsensusBean (consensus_result.rs:37-45) b of a record: rank and identifier at the record's bean level of the bean's
    // first lineage, `taxonomy` that whole lineage
    const blu_bean& bean(const ResultPart& p, const blu_record& rc, uint32_t b) const { return p.beans[rc.bean_base + b]; }
    std::string_view bean_rank(const blu_record& rc, const blu_bean& bn) const { return T.ranks[T.pos_rank[T.lin_off[bn.first_lineage] + rc.bean_level]].full; }
    std::string_view bean_identifier(const blu_record& rc, const blu_bean& bn) const { return T.idents[T.pos_ident[T.lin_off[bn.first_lineage] + rc.bean_level]]; }
    uint32_t occurrences(const blu_bean& bn) const { return bn.occurrences; }
    void append_lineage(std::string& o, const blu_bean& bn) const { T.append_lineage(o, bn.first_lineage); }
    std::string_view accession(const ResultPart& p, const blu_record& rc, const blu_bean& bn, uint32_t a) const {
        const blu_acc& ac = p.accs[rc.acc_base + bn.acc_begin + a];
        return std::string_view(p.pool + BLU_ACC_OFF(ac), BLU_ACC_LEN(ac));
    }

    // ---- serde_json ----
    // `"taxon":{...}` object body in compact or pretty layout
    void taxon(std::string& o, const ResultPart& part, const blu_record& rc, bool pretty, int ind) const {
        auto nl = [&](int extra) {
            if (!pretty) return;
            o.push_back('\n');
            o.append((size_t)(ind + extra) * 2, ' ');
        };
        auto key = [&](int extra, const char* k) {
            nl(extra);
            o.push_back('"');
            o += k;
            o += pretty ? "\": " : "\":";
        };
        std::string& s = scratch();
        o.push_back('{');
        key(1, "reachedRank");
        json_escape(o, reached_rank(rc));
        o.push_back(',');
        key(1, "maxAllowedRank");
        if (const std::string* a = allowed_rank(rc))
            json_escape(o, *a);
        else
            o += "null";
        o.push_back(',');
        key(1, "identifier");
        json_escape(o, identifier(rc));
        o.push_back(',');
        key(1, "percIdentity");
        json_f64(o, rc.perc_identity);
        o.push_back(',');
        key(1, "bitScore");
        json_f64(o, (double)rc.bit_score);
        o.push_back(',');
        key(1, "taxonomy");
        append_taxonomy(s, rc);
        json_escape(o, s);
        o.push_back(',');
        key(1, "mutated");
        o += rc.mutated ? "true," : "false,";
        key(1, "singleMatch");
        o += rc.single_match ? "true," : "false,";
        key(1, "consensusBeans");
        o.push_back('[');
        for (uint32_t b = 0; b < rc.n_beans; b++) {
            const blu_bean& bn = bean(part, rc, b);
            if (b) o.push_back(',');
            nl(2);
            o.push_back('{');
            key(3, "rank");
            json_escape(o, bean_rank(rc, bn));
            o.push_back(',');
            key(3, "identifier");
            json_escape(o, bean_identifier(rc, bn));
            o.push_back(',');
            key(3, "occurrences");
            o += std::to_string(occurrences(bn));
            o.push_back(',');
            key(3, "taxonomy");
            s.clear();
            append_lineage(s, bn);
            json_escape(o, s);
            o.push_back(',');
            key(3, "accessions");
            o.push_back('[');
            for (uint32_t a = 0; a < bn.n_acc; a++) {
                if (a) o.push_back(',');
                nl(4);
                json_escape(o, accession(part, rc, bn, a));
            }
            if (bn.n_acc) nl(3);
            o.push_back(']');
            nl(2);
            o.push_back('}');
        }
        if (rc.n_beans) nl(1);
        o.push_back(']');
        nl(0);
        o.push_back('}');
    }
    // one QueryWithConsensus object (consensus_result.rs:7-13); run_id empty -> field omitted (canonical form)
    void object(std::string& o, std::string_view query, const ResultPart* part, const blu_record* rc, const char* run_id, bool pretty, int ind) const {
        auto nl = [&](int extra) {
            if (!pretty) return;
            o.push_back('\n');
            o.append((size_t)(ind + extra) * 2, ' ');
        };
        const char* colon = pretty ? ": " : ":";
        o.push_back('{');
        if (run_id) {
            nl(1);
            o += "\"runId\"";
            o += colon;
            json_escape(o, run_id);
            o.push_back(',');
        }
        nl(1);
        o += "\"query\"";
        o += colon;
        json_escape(o, query);
        o.push_back(',');
        nl(1);
        o += "\"taxon\"";
        o += colon;
        if (rc)
            taxon(o, *part, *rc, pretty, ind + 1);
        else
            o += "null";
        nl(0);
        o.push_back('}');
    }

    // ---- serde_yaml 0.9: one QueryWithConsensus as an item of the block sequence `results` (write_blutils_output.rs:216-248) ----
    void yaml_object(std::string& o, std::string_view query, const ResultPart* part, const blu_record* rc, std::string_view run_id) const {
        o += "- runId: ";
        yaml_str(o, run_id);
        o += "\n  query: ";
        yaml_str(o, query);
        if (!rc) {
            o += "\n  taxon: null\n";
            return;
        }
        std::string& s = scratch();
        o += "\n  taxon:\n    reachedRank: ";
        yaml_str(o, reached_rank(*rc));
        o += "\n    maxAllowedRank: ";
        if (const std::string* a = allowed_rank(*rc))
            yaml_str(o, *a);
        else
            o += "null";
        o += "\n    identifier: ";
        yaml_str(o, identifier(*rc));
        o += "\n    percIdentity: ";
        yaml_f64(o, rc->perc_identity);
        o += "\n    bitScore: ";
        yaml_f64(o, (double)rc->bit_score);
        o += "\n    taxonomy: ";
        append_taxonomy(s, *rc);
        yaml_str(o, s);
        o += rc->mutated ? "\n    mutated: true" : "\n    mutated: false";
        o += rc->single_match ? "\n    singleMatch: true" : "\n    singleMatch: false";
        o += rc->n_beans ? "\n    consensusBeans:\n" : "\n    consensusBeans: []\n";
        for (uint32_t b = 0; b < rc->n_beans; b++) {
            const blu_bean& bn = bean(*part, *rc, b);
            o += "    - rank: ";
            yaml_str(o, bean_rank(*rc, bn));
            o += "\n      identifier: ";
            yaml_str(o, bean_identifier(*rc, bn));
            o += "\n      occurrences: " + std::to_string(occurrences(bn));
            o += "\n      taxonomy: ";
            s.clear();
            append_lineage(s, bn);
            yaml_str(o, s);
            o += bn.n_acc ? "\n      accessions:\n" : "\n      accessions: []\n";
            for (uint32_t a = 0; a < bn.n_acc; a++) {
                o += "      - ";
                yaml_str(o, accession(*part, *rc, bn, a));
                o.push_back('\n');
            }
        }
    }
};

struct Entry {
    std::string_view query;
    const blu_record* rec;  // nullptr = NoConsensusFound
    const ResultPart* part;
};

// write_blutils_output.rs:87-111 flattens the results: the records of every part in part order, then the hit-less headers
inline std::vector<Entry> all_entries(const ResultView* r) {
    std::vector<Entry> v;
    v.reserve(r->n_rec() + (r->hitless_ ? r->hitless_->size() : 0));
    for (auto& p : r->parts)
        for (uint64_t i = 0; i < p.n_rec; i++) v.push_back({rec_query(p, p.rec[i]), &p.rec[i], &p});
    if (r->hitless_)
        for (auto& h : *r->hitless_) v.push_back({std::string_view(h), nullptr, nullptr});
    return v;
}

inline unsigned host_threads() {
    unsigned n = std::thread::hardware_concurrency();
    return n ? std::min(n, 32u) : 4u;
}

template <class F>
void parallel_ranges(size_t n, F&& f) {
    unsigned nt = (unsigned)std::min<size_t>(host_threads(), std::max<size_t>(1, n / 4096));
    if (nt <= 1) {
        f(0, 0, n);
        return;
    }
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++) th.emplace_back([&, t] { f(t, n * t / nt, n * (t + 1) / nt); });
    for (auto& x : th) x.join();
}

// write_blutils_output.rs:87-111: flatten + sort by query (bytewise).  At 10^6 - 10^8 queries the sort of the ids is what the
// writer waits for first (SURVEY 8f-1): the entries are sorted in per-thread chunks and merged pairwise in parallel (stable:
// equal ids keep their file order, like the reference's sort_by).  Records sorted on the GPU already (ResultView::sorted) are
// only merged with the sorted hit-less headers, records first among equal ids: the same order.
inline std::vector<Entry> sorted_entries(const ResultView* r) {
    std::vector<Entry> v = all_entries(r);
    auto less = [](const Entry& a, const Entry& b) { return a.query < b.query; };
    if (r->sorted) {
        const auto headers = v.begin() + (std::ptrdiff_t)r->n_rec();
        std::stable_sort(headers, v.end(), less);
        std::inplace_merge(v.begin(), headers, v.end(), less);
        return v;
    }
    const size_t n = v.size();
    unsigned nt = (unsigned)std::min<size_t>(host_threads(), std::max<size_t>(1, n / 65536));
    if (nt <= 1) {
        std::stable_sort(v.begin(), v.end(), less);
        return v;
    }
    std::vector<size_t> cut(nt + 1);
    for (unsigned t = 0; t <= nt; t++) cut[t] = n * t / nt;
    {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++) th.emplace_back([&, t] { std::stable_sort(v.begin() + cut[t], v.begin() + cut[t + 1], less); });
        for (auto& x : th) x.join();
    }
    std::vector<Entry> aux(n);
    std::vector<Entry>* src = &v;
    std::vector<Entry>* dst = &aux;
    while (cut.size() > 2) {
        std::vector<size_t> ncut;
        std::vector<std::thread> th;
        for (size_t i = 0; i + 1 < cut.size(); i += 2) {
            ncut.push_back(cut[i]);
            if (i + 2 < cut.size()) {
                const size_t a = cut[i], m = cut[i + 1], b = cut[i + 2];
                th.emplace_back([=] { std::merge(src->begin() + a, src->begin() + m, src->begin() + m, src->begin() + b, dst->begin() + a, less); });
            } else {
                const size_t a = cut[i], b = cut[i + 1];
                th.emplace_back([=] { std::copy(src->begin() + a, src->begin() + b, dst->begin() + a); });
            }
        }
        ncut.push_back(n);
        for (auto& x : th) x.join();
        cut.swap(ncut);
        std::swap(src, dst);
    }
    if (src != &v) v.swap(aux);
    return v;
}

// Formats entries [0, n) with `emit(out, i)` on all host threads, blocks of entries at a time.  To a regular file every
// thread writes its own blocks with pwrite() at the offset its predecessors' sizes give it (the copy into the page cache is
// what a single writer thread is bound by: ~2 GB/s); to a pipe / terminal the blocks are written in order by the caller's
// thread while later ones are still being formatted.  Returns false on a write error.
template <class Emit>
bool ordered_parallel_write(FILE* f, size_t n, Emit&& emit) {
    const size_t B = 4096;
    const size_t nblocks = (n + B - 1) / B;
    const unsigned nt = (unsigned)std::min<size_t>(host_threads(), nblocks);
    if (nt <= 1 || nblocks < 4) {
        std::string o;
        bool ok = true;
        for (size_t i = 0; i < n; i++) {
            emit(o, i);
            if (o.size() > (8u << 20)) {
                ok &= fwrite(o.data(), 1, o.size(), f) == o.size();
                o.clear();
            }
        }
        ok &= fwrite(o.data(), 1, o.size(), f) == o.size();
        return ok;
    }
    fflush(f);
    const int fd = fileno(f);
    struct stat st;
    const bool seekable = fd >= 0 && fstat(fd, &st) == 0 && S_ISREG(st.st_mode);
    std::atomic<size_t> next{0};
    std::atomic<bool> failed{false};
    if (seekable) {
        const long long base_off = (long long)ftello(f);
        std::unique_ptr<std::atomic<long long>[]> end_off(new std::atomic<long long>[nblocks]);
        for (size_t b = 0; b < nblocks; b++) end_off[b].store(-1);
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++)
            th.emplace_back([&] {
                std::string o;
                for (;;) {
                    const size_t b = next.fetch_add(1);
                    if (b >= nblocks) return;
                    o.clear();
                    o.reserve(B * 512);
                    const size_t e = std::min(n, (b + 1) * B);
                    for (size_t i = b * B; i < e; i++) emit(o, i);
                    long long off = base_off;
                    if (b) {
                        while ((off = end_off[b - 1].load(std::memory_order_acquire)) < 0) std::this_thread::yield();
                    }
                    end_off[b].store(off + (long long)o.size(), std::memory_order_release);
                    size_t done = 0;
                    while (done < o.size()) {
                        const ssize_t w = pwrite(fd, o.data() + done, o.size() - done, (off_t)(off + (long long)done));
                        if (w < 0 && errno == EINTR) continue;
                        if (w <= 0) {
                            failed = true;
                            break;
                        }
                        done += (size_t)w;
                    }
                }
            });
        for (auto& x : th) x.join();
        if (failed) return false;
        return fseeko(f, (off_t)end_off[nblocks - 1].load(), SEEK_SET) == 0;
    }
    std::vector<std::string> out(nblocks);
    std::unique_ptr<std::atomic<int>[]> ready(new std::atomic<int>[nblocks]);
    for (size_t b = 0; b < nblocks; b++) ready[b].store(0);
    std::atomic<size_t> written{0};
    const size_t window = 4 * (size_t)nt;  // blocks formatted ahead of the writer: bounds the memory
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++)
        th.emplace_back([&] {
            for (;;) {
                const size_t b = next.fetch_add(1);
                if (b >= nblocks) return;
                while (b >= written.load(std::memory_order_acquire) + window) std::this_thread::yield();
                std::string& o = out[b];
                o.reserve(B * 512);
                const size_t e = std::min(n, (b + 1) * B);
                for (size_t i = b * B; i < e; i++) emit(o, i);
                ready[b].store(1, std::memory_order_release);
            }
        });
    bool ok = true;
    for (size_t b = 0; b < nblocks; b++) {
        while (!ready[b].load(std::memory_order_acquire)) std::this_thread::yield();
        ok &= fwrite(out[b].data(), 1, out[b].size(), f) == out[b].size();
        std::string().swap(out[b]);
        written.store(b + 1, std::memory_order_release);
    }
    for (auto& x : th) x.join();
    return ok;
}

inline std::string uuid_v4() {
    std::random_device rd;
    uint8_t b[16];
    for (int i = 0; i < 16; i += 4) {
        uint32_t x = rd();
        memcpy(b + i, &x, 4);
    }
    b[6] = (b[6] & 0x0F) | 0x40;
    b[8] = (b[8] & 0x3F) | 0x80;
    char s[40];
    snprintf(s, sizeof s, "%02x%02x%02x%02x-%02x%02x-%02x%02x-%02x%02x-%02x%02x%02x%02x%02x%02x", b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7],
             b[8], b[9], b[10], b[11], b[12], b[13], b[14], b[15]);
    return s;
}

// serde_yaml 0.9 string scalars (write_blutils_output.rs:216-248 serialises with serde_yaml::to_writer).  The crate is
// not vendored under /root/reference: restated from its published behaviour (PARITY UNPINNED; the test oracle holds an
// independent statement of the same rules, tests/test_yaml_scalars.py compares the two byte for byte):
//   * single-quoted when the string would read back as another type (serde_yaml ser.rs serialize_str -> de.rs
//     visit_untagged_scalar): empty, null / ~, true / false, integers (also 0x / 0o / 0b), floats (also .inf / .nan), or is a
//     YAML 1.1 boolean (y, yes, n, no, on, off, any case);
//   * else libyaml's emitter (yaml_emitter_analyze_scalar / select_scalar_style, block context): plain unless there is a
//     leading / trailing space, a non-printable character, a leading indicator, "- " / "? " / ": " at the start, "---" / "...",
//     ": " / trailing ":" / " #" inside; then single-quoted, double-quoted only for non-printable characters.
inline bool yaml_digits_but_not_number(std::string_view s) {
    if (!s.empty() && (s[0] == '+' || s[0] == '-')) s.remove_prefix(1);
    if (s.size() <= 1 || s[0] != '0') return false;
    for (size_t i = 1; i < s.size(); i++)
        if (s[i] < '0' || s[i] > '9') return false;
    return true;
}

inline bool yaml_fits_u128(std::string_view digits, int radix) {  // value of a valid digit string < 2^128
    unsigned __int128 v = 0;
    for (char ch : digits) {
        const int d = ch <= '9' ? ch - '0' : (ch | 0x20) - 'a' + 10;
        const unsigned __int128 lim = ~(unsigned __int128)0;
        if (v > (lim - (unsigned)d) / (unsigned)radix) return false;
        v = v * (unsigned)radix + (unsigned)d;
    }
    return true;
}

inline bool yaml_int_like(std::string_view s) {
    std::string_view body = s;
    if (!body.empty() && (body[0] == '+' || body[0] == '-')) body.remove_prefix(1);
    if (body.empty() || body[0] == '+' || body[0] == '-') return false;
    if (body.size() >= 2 && body[0] == '0' && (body[1] == 'x' || body[1] == 'o' || body[1] == 'b')) {
        const int radix = body[1] == 'x' ? 16 : body[1] == 'o' ? 8 : 2;
        std::string_view rest = body.substr(2);
        if (rest.empty()) return false;
        for (char ch : rest) {
            const bool ok = radix == 16 ? ((ch >= '0' && ch <= '9') || ((ch | 0x20) >= 'a' && (ch | 0x20) <= 'f')) : (ch >= '0' && ch < '0' + radix);
            if (!ok) return false;
        }
        return yaml_fits_u128(rest, radix);
    }
    if (yaml_digits_but_not_number(s)) return false;
    for (char ch : body)
        if (ch < '0' || ch > '9') return false;
    return yaml_fits_u128(body, 10);
}

inline bool yaml_float_like(std::string_view s) {
    if (yaml_digits_but_not_number(s)) return false;
    std::string_view u = s;
    if (!u.empty() && u[0] == '+') {
        u.remove_prefix(1);
        if (!u.empty() && (u[0] == '+' || u[0] == '-')) return false;
    }
    if (u == ".inf" || u == ".Inf" || u == ".INF" || s == "-.inf" || s == "-.Inf" || s == "-.INF" || s == ".nan" || s == ".NaN" || s == ".NAN") return true;
    // [+-]? (digits [. digits*] | . digits+) ([eE] [+-]? digits+)?
    size_t i = 0;
    if (i < u.size() && (u[i] == '+' || u[i] == '-')) i++;
    size_t nint = 0, nfrac = 0;
    while (i < u.size() && u[i] >= '0' && u[i] <= '9') i++, nint++;
    if (i < u.size() && u[i] == '.') {
        i++;
        while (i < u.size() && u[i] >= '0' && u[i] <= '9') i++, nfrac++;
    }
    if (nint == 0 && nfrac == 0) return false;
    if (i < u.size() && (u[i] == 'e' || u[i] == 'E')) {
        i++;
        if (i < u.size() && (u[i] == '+' || u[i] == '-')) i++;
        size_t nexp = 0;
        while (i < u.size() && u[i] >= '0' && u[i] <= '9') i++, nexp++;
        if (nexp == 0) return false;
    }
    if (i != u.size()) return false;
    const std::string z(u);
    char* end = nullptr;
    const double v = strtod(z.c_str(), &end);
    return v - v == 0.0;  // finite (an overflowing literal reads back as a string)
}

inline bool yaml_printable(uint32_t cp) {
    return cp == 0x0A || (cp >= 0x20 && cp <= 0x7E) || cp == 0x85 || (cp >= 0xA0 && cp <= 0xD7FF) || (cp >= 0xE000 && cp <= 0xFFFD && cp != 0xFEFF) ||
           (cp >= 0x10000 && cp <= 0x10FFFF);
}

// next code point of a UTF-8 string (malformed bytes are returned as themselves, one at a time: they are not printable)
inline uint32_t yaml_next_cp(std::string_view s, size_t& i) {
    const unsigned char c = (unsigned char)s[i];
    auto cont = [&](size_t k) { return i + k < s.size() && ((unsigned char)s[i + k] & 0xC0) == 0x80; };
    if (c < 0x80) return i += 1, c;
    if ((c & 0xE0) == 0xC0 && cont(1)) {
        const uint32_t cp = ((c & 0x1Fu) << 6) | ((unsigned char)s[i + 1] & 0x3Fu);
        return i += 2, cp;
    }
    if ((c & 0xF0) == 0xE0 && cont(1) && cont(2)) {
        const uint32_t cp = ((c & 0x0Fu) << 12) | (((unsigned char)s[i + 1] & 0x3Fu) << 6) | ((unsigned char)s[i + 2] & 0x3Fu);
        return i += 3, cp;
    }
    if ((c & 0xF8) == 0xF0 && cont(1) && cont(2) && cont(3)) {
        const uint32_t cp = ((c & 0x07u) << 18) | (((unsigned char)s[i + 1] & 0x3Fu) << 12) | (((unsigned char)s[i + 2] & 0x3Fu) << 6) | ((unsigned char)s[i + 3] & 0x3Fu);
        return i += 4, cp;
    }
    return i += 1, (uint32_t)c | 0x80000000u;
}

inline void yaml_str(std::string& o, std::string_view s) {
    auto single = [&]() {
        o.push_back('\'');
        for (char ch : s) {
            if (ch == '\'') o.push_back('\'');
            o.push_back(ch);
        }
        o.push_back('\'');
    };
    std::string lower(s);
    for (char& ch : lower)
        if (ch >= 'A' && ch <= 'Z') ch = (char)(ch + 32);
    static const char* ambiguous[] = {"y", "yes", "n", "no", "on", "off", "true", "false", "null", "~"};
    bool amb = s.empty();
    for (auto a : ambiguous) amb |= lower == a;
    if (amb || yaml_int_like(s) || yaml_float_like(s)) return single();
    bool special = false;
    for (size_t i = 0; i < s.size();) {
        const uint32_t cp = yaml_next_cp(s, i);
        special |= !yaml_printable(cp) || cp == 0x0A;
    }
    if (special) {
        o.push_back('"');
        for (size_t i = 0; i < s.size();) {
            const size_t at = i;
            const uint32_t cp = yaml_next_cp(s, i);
            const bool esc = !yaml_printable(cp) || cp == 0xFEFF || cp == 0x0A || cp == 0x0D || cp == 0x85 || cp == 0x2028 || cp == 0x2029 || cp == '"' || cp == '\\';
            if (!esc) {
                o.append(s.substr(at, i - at));
                continue;
            }
            switch (cp) {
                case 0: o += "\\0"; break;
                case 7: o += "\\a"; break;
                case 8: o += "\\b"; break;
                case 9: o += "\\t"; break;
                case 10: o += "\\n"; break;
                case 11: o += "\\v"; break;
                case 12: o += "\\f"; break;
                case 13: o += "\\r"; break;
                case 27: o += "\\e"; break;
                case '"': o += "\\\""; break;
                case '\\': o += "\\\\"; break;
                case 0x85: o += "\\N"; break;
                case 0xA0: o += "\\_"; break;
                case 0x2028: o += "\\L"; break;
                case 0x2029: o += "\\P"; break;
                default: {
                    char b[16];
                    const uint32_t v = cp & 0x7FFFFFFFu;
                    if (v <= 0xFF)
                        snprintf(b, sizeof b, "\\x%02X", v);
                    else if (v <= 0xFFFF)
                        snprintf(b, sizeof b, "\\u%04X", v);
                    else
                        snprintf(b, sizeof b, "\\U%08X", v);
                    o += b;
                }
            }
        }
        o.push_back('"');
        return;
    }
    bool block_ind = s.substr(0, 3) == "---" || s.substr(0, 3) == "...";
    for (size_t i = 0; i < s.size(); i++) {
        const char c = s[i];
        const bool nxt_blank = i + 1 >= s.size() || s[i + 1] == ' ' || s[i + 1] == '\t';
        if (i == 0) {
            if (strchr("#,[]{}&*!|>'\"%@`", c)) block_ind = true;
            if ((c == '?' || c == ':' || c == '-') && nxt_blank) block_ind = true;
        } else {
            if (c == ':' && nxt_blank) block_ind = true;
            if (c == '#' && (s[i - 1] == ' ' || s[i - 1] == '\t')) block_ind = true;
        }
    }
    if (block_ind || s.front() == ' ' || s.back() == ' ') return single();
    o.append(s);
}

inline void yaml_f64(std::string& o, double v) {  // serde_yaml: ryu, but integers print without ".0"?  No: serde_yaml keeps ryu's output
    json_f64(o, v);
}

inline uint64_t view_checksum(const ResultView* r) {
    Decoder d(r);
    std::atomic<uint64_t> total{0};
    auto fnv = [](const std::string& s) {
        uint64_t h = 0xcbf29ce484222325ull;
        for (unsigned char ch : s) {
            h ^= ch;
            h *= 0x100000001b3ull;
        }
        return h;
    };
    for (auto& p : r->parts)
        parallel_ranges(p.n_rec, [&](unsigned, size_t a, size_t b) {
            std::string line;
            uint64_t sum = 0;
            for (size_t i = a; i < b; i++) {
                line.clear();
                d.object(line, rec_query(p, p.rec[i]), &p, &p.rec[i], nullptr, false, 0);
                sum += fnv(line);
            }
            total += sum;
        });
    if (r->hitless_)
        for (auto& h : *r->hitless_) {
            std::string line;
            d.object(line, h, nullptr, nullptr, nullptr, false, 0);
            total += fnv(line);
        }
    return total.load();
}


// `max_entries` < number of entries: only the entries with the smallest query ids (partial sort), in order
inline std::string view_to_jsonl(const ResultView* r, uint64_t max_entries = ~0ull) {
    Decoder d(r);
    std::vector<Entry> ent;
    const uint64_t total = r->n_rec() + (r->hitless_ ? r->hitless_->size() : 0);
    if (max_entries < total && !r->sorted) {
        ent = all_entries(r);
        // (ties keep their file order like the stable full sort: compare the position as the last key)
        std::vector<uint64_t> idx(total);
        for (uint64_t i = 0; i < total; i++) idx[i] = i;
        std::partial_sort(idx.begin(), idx.begin() + (std::ptrdiff_t)max_entries, idx.end(), [&](uint64_t a, uint64_t b) {
            const int c = ent[a].query.compare(ent[b].query);
            return c != 0 ? c < 0 : a < b;
        });
        std::vector<Entry> head;
        head.reserve(max_entries);
        for (uint64_t i = 0; i < max_entries; i++) head.push_back(ent[idx[i]]);
        ent.swap(head);
    } else {
        ent = sorted_entries(r);
        if (ent.size() > max_entries) ent.resize(max_entries);
    }
    std::vector<std::string> parts(host_threads());
    parallel_ranges(ent.size(), [&](unsigned t, size_t a, size_t b) {
        std::string& o = parts[t];
        for (size_t i = a; i < b; i++) {
            d.object(o, ent[i].query, ent[i].part, ent[i].rec, nullptr, false, 0);
            o.push_back('\n');
        }
    });
    size_t tot = 0;
    for (auto& p : parts) tot += p.size();
    std::string out;
    out.reserve(tot);
    for (auto& p : parts) out += p;
    return out;
}

// write_blutils_output.rs:42-52: the extension is forced to match the format (the last dot after the last '/' starts it)
inline std::string with_extension(const char* path, const char* ext) {
    std::string target = path;
    const size_t slash = target.find_last_of('/');
    const size_t dot = target.find_last_of('.');
    if (dot != std::string::npos && (slash == std::string::npos || dot > slash)) target.resize(dot);
    return target + ext;
}

inline int view_write(const ResultView* r, const char* path, int format, const char* run_id_in) {
    Decoder d(r);
    auto ent = sorted_entries(r);
    const std::string run_id = run_id_in ? std::string(run_id_in) : uuid_v4();
    FILE* f = stdout;
    if (path) {
        const std::string target = with_extension(path, format == BLU_FORMAT_JSON ? ".json" : format == BLU_FORMAT_JSONL ? ".jsonl" : ".yaml");
        {
            std::error_code ec;
            auto parent = std::filesystem::path(target).parent_path();
            if (!parent.empty()) std::filesystem::create_directories(parent, ec);  // write_blutils_output.rs:64-73
        }
        f = fopen(target.c_str(), "wb");
        if (!f) return BLU_ERR_IO;
    }
    const bool pretty = format == BLU_FORMAT_JSON && path != nullptr;  // to_string_pretty to a file, compact to stdout
    bool wok = true;
    auto put = [&](const char* t) { fwrite(t, 1, strlen(t), f); };
    if (format == BLU_FORMAT_JSON) {
        put(pretty ? "{\n  \"results\": [" : "{\"results\":[");
        wok &= ordered_parallel_write(f, ent.size(), [&](std::string& o, size_t i) {
            if (i) o.push_back(',');
            if (pretty) o += "\n    ";
            d.object(o, ent[i].query, ent[i].part, ent[i].rec, run_id.c_str(), pretty, 2);
        });
        if (pretty)
            put(ent.empty() ? "],\n  \"config\": null\n}" : "\n  ],\n  \"config\": null\n}");
        else
            put("],\"config\":null}");
    } else if (format == BLU_FORMAT_JSONL) {
        put("null\n");  // serde_json::to_string(&config) with config = None
        wok &= ordered_parallel_write(f, ent.size(), [&](std::string& o, size_t i) {
            d.object(o, ent[i].query, ent[i].part, ent[i].rec, run_id.c_str(), false, 0);
            o.push_back('\n');
        });
    } else {
        // serde_yaml 0.9 block style of BlutilsOutput{results, config}
        put(ent.empty() ? "results: []\n" : "results:\n");
        wok &= ordered_parallel_write(f, ent.size(), [&](std::string& o, size_t i) { d.yaml_object(o, ent[i].query, ent[i].part, ent[i].rec, run_id); });
        put("config: null\n");
    }
    if (path)
        wok &= fclose(f) == 0;
    else
        fflush(stdout);
    return wok ? BLU_OK : BLU_ERR_IO;
}


// ---------------------------------------------------------------------------------------------------------------
// build-tabular: the 12-column TSV of parse_consensus_as_tabular (reference core/src/use_cases/parse_consensus_as_tabular/
// mod.rs:15-173), for the records (view_write_tabular) and for a result file (result_file_to_tabular, blu_tabular.h).
// Byte-exact quirks kept:
//   * to stdout every piece goes through println! (one '\n' each), so a query without taxon, whose piece already ends
//     in '\n', is followed by an empty line;
//   * to a file the pieces are written as they are -- the reference never adds the line breaks there (mod.rs:58-66 +
//     shared/write_file_or_stdout.rs), so only the taxon-less pieces end a line;
//   * floats use Rust's Display (845.0 -> "845").
// The header and every piece after it are followed by tsv_end_piece.
// ---------------------------------------------------------------------------------------------------------------
inline void tsv_end_piece(std::string& o, bool to_stdout) {
    if (to_stdout) o.push_back('\n');
}

inline void tsv_header(std::string& o) {
    o += "run-id\tquery\ttype\trank\tidentifier\tperc-identity\tbit-score\ttaxonomy\tmutated\tsingle-match\toccurrences\taccessions";
}

// a query without taxon: no run id, no other column
inline void tsv_no_taxon(std::string& o, std::string_view query) {
    o.append(query);
    o += "\tnull\n";
}

inline void tsv_consensus(std::string& o, std::string_view run_id, std::string_view query, std::string_view rank, std::string_view identifier,
                          double perc_identity, double bit_score, std::string_view taxonomy, bool mutated, bool single_match) {
    o.append(run_id);
    o.push_back('\t');
    o.append(query);
    o += "\tconsensus\t";
    o.append(rank);
    o.push_back('\t');
    o.append(identifier);
    o.push_back('\t');
    rust_display_f64(o, perc_identity);
    o.push_back('\t');
    rust_display_f64(o, bit_score);
    o.push_back('\t');
    o.append(taxonomy);
    o += mutated ? "\ttrue" : "\tfalse";
    o += single_match ? "\ttrue" : "\tfalse";
    o += "\tnull\tnull";
}

// one consensus bean, up to the accessions column; the caller then appends every accession with tsv_accession.  bit_score is
// the taxon's.
inline void tsv_blast_match(std::string& o, std::string_view run_id, std::string_view query, std::string_view rank, std::string_view identifier,
                            double bit_score, std::string_view taxonomy, int64_t occurrences) {
    o.append(run_id);
    o.push_back('\t');
    o.append(query);
    o += "\tblast-match\t";
    o.append(rank);
    o.push_back('\t');
    o.append(identifier);
    o += "\tnull\t";
    rust_display_f64(o, bit_score);
    o.push_back('\t');
    o.append(taxonomy);
    o += "\tnull\tnull\t";
    o += std::to_string(occurrences);
    o.push_back('\t');
}

inline void tsv_accession(std::string& o, size_t i, std::string_view accession) {
    if (i) o += ", ";
    o.append(accession);
}

// The TSV straight from the binary records instead of re-reading the JSON.
inline int view_write_tabular(const ResultView* r, const char* path, const char* run_id_in) {
    Decoder d(r);
    auto ent = sorted_entries(r);
    const std::string run_id = run_id_in ? std::string(run_id_in) : uuid_v4();
    const bool to_stdout = path == nullptr;
    FILE* f = stdout;
    if (path) {
        const std::string target = with_extension(path, ".tsv");
        std::remove(target.c_str());
        f = fopen(target.c_str(), "wb");  // (the reference appends to a file it has just removed; pwrite needs a non-append descriptor)
        if (!f) return BLU_ERR_IO;
    }
    {
        std::string h;
        tsv_header(h);
        tsv_end_piece(h, to_stdout);
        fwrite(h.data(), 1, h.size(), f);
    }
    const bool ok = ordered_parallel_write(f, ent.size(), [&](std::string& o, size_t ei) {
        const Entry& en = ent[ei];
        if (!en.rec) {
            tsv_no_taxon(o, en.query);
            tsv_end_piece(o, to_stdout);
            return;
        }
        const blu_record& rc = *en.rec;
        std::string& s = scratch();
        d.append_taxonomy(s, rc);
        tsv_consensus(o, run_id, en.query, d.reached_rank(rc), d.identifier(rc), rc.perc_identity, (double)rc.bit_score, s, rc.mutated, rc.single_match);
        tsv_end_piece(o, to_stdout);
        for (uint32_t b = 0; b < rc.n_beans; b++) {
            const blu_bean& bn = d.bean(*en.part, rc, b);
            s.clear();
            d.append_lineage(s, bn);
            tsv_blast_match(o, run_id, en.query, d.bean_rank(rc, bn), d.bean_identifier(rc, bn), (double)rc.bit_score, s, d.occurrences(bn));
            for (uint32_t a = 0; a < bn.n_acc; a++) tsv_accession(o, a, d.accession(*en.part, rc, bn, a));
            tsv_end_piece(o, to_stdout);
        }
    });
    if (path)
        fclose(f);
    else
        fflush(stdout);
    return ok ? BLU_OK : BLU_ERR_IO;
}

}  // namespace blu
