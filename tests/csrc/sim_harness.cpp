// TEST INFRASTRUCTURE ONLY -- host simulation of the device-side logic.
// Compiles blutils_b200/csrc/blu_core.cuh (the `__host__ __device__` parsing / join / consensus code the CUDA
// kernels call), blu_taxonomy.cpp and blu_decode.h with g++ and drives them with a trivial sequential loop, so
// that the per-row and per-query logic can be checked against the oracle on a machine without a GPU.
// It is NOT linked into libblu_consensus.so and is not a fallback: the kernel-side control flow (windows, row
// index, run ownership, deferral, streaming) only exists in blu_kernels.cu and is tested on the GPU.
#include <cstdlib>
#include <cstring>
#include <string>
#include <functional>
#include <unordered_set>
#include <vector>

#include "../../blutils_b200/csrc/blu_core.cuh"
#include "../../blutils_b200/csrc/blu_decode.h"
#include "../../blutils_b200/csrc/blu_taxonomy.h"

using namespace blu;

static int map_err(uint32_t e) {
    if (e == DE_NONE) return BLU_OK;
    if (e >= DE_INTERNAL) return BLU_ERR_INTERNAL;
    if (e >= DE_NUM_UNSUPPORTED) return BLU_ERR_UNSUPPORTED;
    return BLU_ERR_DATA;
}

// The path on the host (device core + host taxonomy build), the finished result handed to `emit`.
static int sim_run_impl(const int64_t* taxids, const uint64_t* off, const char* blob, uint64_t n, int taxon, int has_custom, const int32_t* custom8,
                        int strategy, const char* text, uint64_t nbytes, const char* headers_nl, uint64_t headers_len,
                        const std::function<void(const ResultView&)>& emit, char* err, int errlen) {
    try {
        Cutoffs cut;
        cut.taxon = taxon;
        cut.has_custom = has_custom != 0;
        if (has_custom)
            for (int i = 0; i < 8; i++) cut.custom[i] = custom8[i];
        HostTaxonomy T;
        build_taxonomy(taxids, off, blob, n, cut, T);
        LinTables L{};
        L.lin_off = T.lin_off.data();
        L.lvl_key = T.lvl_key.data();
        L.bean_key = T.bean_key.data();
        L.ident_rank = T.ident_rank.data();
        L.cut = T.cut.data();
        L.rank_cls = T.rank_cls.data();
        L.allowed_cls = T.allowed_cls.data();
        L.lin_ok = T.lin_ok.data();
        L.slots = T.slots.data();
        L.hash_mask = T.hash_mask;
        L.n_lin = (uint32_t)T.n_lin();
        if (nbytes == 0) throw DataErr("empty blast output");
        const uint8_t* tx = (const uint8_t*)text;
        struct R {
            uint64_t s;
            int len;
            int64_t bits;
            int qlen;
        };
        std::vector<R> rows;
        long n_fast = 0, n_lean = 0, n_info = 0;
        // byte-class bitmasks exactly as the row scan of the kernels publishes them (bit i = byte i)
        std::vector<uint64_t> tabw(nbytes / 64 + 3, 0), digw(nbytes / 64 + 3, 0);
        for (uint64_t i = 0; i < nbytes; i++) {
            if (tx[i] == '\t') tabw[i >> 6] |= 1ull << (i & 63);
            if (tx[i] >= '0' && tx[i] <= '9') digw[i >> 6] |= 1ull << (i & 63);
            if (tx[i] == '"' || tx[i] == '\r') {
                snprintf(err, errlen, "device error %u at byte %llu", (unsigned)DE_QUOTE_OR_CR, (unsigned long long)i);
                return map_err(DE_QUOTE_OR_CR);
            }
        }
        if (nbytes > 0x7fffff00ull) throw std::invalid_argument("sim: text too large");
        for (uint64_t p = 0; p < nbytes;) {
            const void* nl = memchr(tx + p, '\n', nbytes - p);
            uint64_t e = nl ? (uint64_t)((const uint8_t*)nl - tx) : nbytes;
            if (e > p) {
                LightRow lr = parse_row_masked(tx, tabw.data(), digw.data(), (int)p, (int)e);
                {
                    // the register fast path may only accept rows the full parser accepts, with identical outputs
                    int64_t fb = 0;
                    int fq = 0;
                    if (parse_row_fast(tx, reinterpret_cast<const uint32_t*>(tabw.data()), reinterpret_cast<const uint32_t*>(digw.data()), (int)p, (int)e,
                                       fb, fq)) {
                        n_fast++;
                        if (lr.err || fb != lr.bits || fq != lr.q_len) {
                            snprintf(err, errlen, "fast row parser disagrees with the full parser at byte %llu", (unsigned long long)p);
                            return BLU_ERR_INTERNAL;
                        }
                    }
                }
                {
                    // same contract for the streaming kernel's lean parser
                    int64_t fb = 0;
                    int fq = 0;
                    uint32_t info = 0;
                    if (parse_row_lean(tx, reinterpret_cast<const uint32_t*>(tabw.data()), reinterpret_cast<const uint32_t*>(digw.data()), (int)p, (int)e,
                                       fb, fq, info)) {
                        n_lean++;
                        if (lr.err || fb != lr.bits || fq != lr.q_len) {
                            snprintf(err, errlen, "lean row parser disagrees with the full parser at byte %llu", (unsigned long long)p);
                            return BLU_ERR_INTERNAL;
                        }
                        {
                            // the tab positions it hands over must split the row like the full splitter does
                            TopRowRaw ra, rb;
                            if (top_row_from_info(tx, (int)p, info, 0, ra)) {
                                n_info++;
                                const uint32_t eb = split_top_row(tx, tabw.data(), (int)p, (int)e, 0, rb);
                                if (eb || ra.acc_off != rb.acc_off || ra.acc_len != rb.acc_len || ra.taxid != rb.taxid || ra.alnlen != rb.alnlen ||
                                    toprow_pident(ra) != toprow_pident(rb)) {
                                    snprintf(err, errlen, "row info of the lean parser splits the row differently at byte %llu", (unsigned long long)p);
                                    return BLU_ERR_INTERNAL;
                                }
                            }
                        }
                    }
                }
                LightRow l2 = light_parse_row(tx + p, (int)(e - p));  // byte-wise variant must agree
                if ((lr.err != 0) != (l2.err != 0) || (!lr.err && (lr.bits != l2.bits || lr.q_len != l2.q_len))) {
                    snprintf(err, errlen, "masked and byte-wise row parsers disagree at byte %llu", (unsigned long long)p);
                    return BLU_ERR_INTERNAL;
                }
                if (lr.err) {
                    snprintf(err, errlen, "device error %u at byte %llu", lr.err, (unsigned long long)p);
                    return map_err(lr.err);
                }
                rows.push_back({p, (int)(e - p), lr.bits, lr.q_len});
            }
            p = e + 1;
        }
        if (rows.empty()) throw DataErr("no rows");
        if (getenv("BLU_SIM_VERBOSE")) fprintf(stderr, "sim: %zu rows, %ld through the fast row parser, %ld through the lean one, %ld with usable tab positions\n", rows.size(), n_fast, n_lean, n_info);
        std::vector<blu_record> recs;
        std::vector<blu_bean> beans;
        std::vector<blu_acc> accs;
        std::unordered_set<std::string> seen;
        std::vector<TopRow> top;
        std::vector<uint16_t> scratch;
        for (size_t h = 0; h < rows.size();) {
            size_t e = h + 1;
            while (e < rows.size()) {
                const bool same = same_first_field(tx, tabw.data(), (int)rows[e - 1].s, (int)rows[e - 1].s + rows[e - 1].len, (int)rows[e].s,
                                                   (int)rows[e].s + rows[e].len);
                // the streaming kernel's variant (knows the id length of the current row) must agree
                if (same_qid_lean(tx, reinterpret_cast<const uint32_t*>(tabw.data()), (int)rows[e].s, rows[e].qlen, (int)rows[e - 1].s) != same) {
                    snprintf(err, errlen, "lean query-id compare disagrees at byte %llu", (unsigned long long)rows[e].s);
                    return BLU_ERR_INTERNAL;
                }
                if (!same) break;
                e++;
            }
            if (!seen.insert(std::string((const char*)tx + rows[h].s, rows[h].qlen)).second) {
                snprintf(err, errlen, "non-contiguous query");
                return BLU_ERR_UNSUPPORTED;
            }
            int64_t mx = rows[h].bits;
            for (size_t r = h; r < e; r++) mx = std::max(mx, rows[r].bits);
            top.clear();
            for (size_t r = h; r < e; r++)
                if (rows[r].bits == mx) {
                    TopRow t;
                    // the kernels' path: field split + number parse (tile kernel), then the taxid join (consensus kernel)
                    TopRowRaw raw;
                    uint32_t er = split_top_row(tx, tabw.data(), (int)rows[r].s, (int)rows[r].s + rows[r].len, 0, raw);
                    if (!er) er = join_top_row(raw, L, t);
                    {
                        TopRow t2;
                        uint32_t er2 = heavy_parse_row(tx + rows[r].s, rows[r].len, rows[r].s, L, t2);
                        if (er != er2 || (!er && (t.acc_off != t2.acc_off || t.acc_len != t2.acc_len || t.lin != t2.lin || t.pident != t2.pident ||
                                                  t.alnlen != t2.alnlen || t.lin_len != t2.lin_len))) {
                            snprintf(err, errlen, "masked and byte-wise top-row parsers disagree at byte %llu", (unsigned long long)rows[r].s);
                            return BLU_ERR_INTERNAL;
                        }
                    }
                    if (er) {
                        snprintf(err, errlen, "device error %u at byte %llu", er, (unsigned long long)rows[r].s);
                        return map_err(er);
                    }
                    top.push_back(t);
                }
            const size_t g = top.size();
            if (g > 65535) return BLU_ERR_UNSUPPORTED;
            blu_record rec = record_header(rows[h].s, (uint32_t)rows[h].qlen, (uint32_t)(e - h), mx);
            rec.bean_base = (uint32_t)beans.size();
            rec.acc_base = (uint32_t)accs.size();
            beans.resize(beans.size() + g);
            accs.resize(accs.size() + g);
            scratch.assign(5 * g, 0);
            QueryOut qo{&rec, beans.data() + rec.bean_base, accs.data() + rec.acc_base};
            uint32_t ce = g == 1 ? consensus_single(top[0], L, qo) : consensus_multi(top.data(), (int)g, tx, L, strategy, scratch.data(), qo);
            if (ce) {
                snprintf(err, errlen, "device error %u in query at byte %llu", ce, (unsigned long long)rows[h].s);
                return map_err(ce);
            }
            recs.push_back(rec);
            h = e;
        }
        std::vector<std::string> hitless;
        if (headers_nl) {
            std::unordered_set<std::string> have;
            for (auto& rc : recs) have.insert(std::string(text + rc.query_off, rc.query_len));
            const char* p = headers_nl;
            const char* e = headers_nl + headers_len;
            while (p < e) {
                const char* nl = (const char*)memchr(p, '\n', e - p);
                const char* le = nl ? nl : e;
                std::string hd(p, le - p);
                if (!have.count(hd)) hitless.push_back(hd);
                p = le + 1;
            }
        }
        ResultView v;
        v.tax = &T;
        v.cut = cut;
        ResultPart part;
        part.rec = recs.data();
        part.beans = beans.data();
        part.accs = accs.data();
        part.pool = text;
        part.n_rec = recs.size();
        v.parts.push_back(part);
        v.hitless_ = &hitless;
        emit(v);
        return BLU_OK;
    } catch (const DataErr& e) {
        snprintf(err, errlen, "%s", e.what());
        return BLU_ERR_DATA;
    } catch (const std::invalid_argument& e) {
        snprintf(err, errlen, "%s", e.what());
        return BLU_ERR_UNSUPPORTED;
    } catch (const std::exception& e) {
        snprintf(err, errlen, "%s", e.what());
        return BLU_ERR_INTERNAL;
    }
}

extern "C" int blu_sim_run(const int64_t* taxids, const uint64_t* off, const char* blob, uint64_t n, int taxon, int has_custom,
                           const int32_t* custom8, int strategy, const char* text, uint64_t nbytes, const char* headers_nl, uint64_t headers_len,
                           char** out, uint64_t* out_len, char* err, int errlen) {
    return sim_run_impl(taxids, off, blob, n, taxon, has_custom, custom8, strategy, text, nbytes, headers_nl, headers_len,
                        [&](const ResultView& v) {
                            std::string js = view_to_jsonl(&v);
                            *out = (char*)malloc(js.size() + 1);
                            memcpy(*out, js.data(), js.size());
                            (*out)[js.size()] = 0;
                            *out_len = js.size();
                        },
                        err, errlen);
}

// Same, the result written by the product's writers (blu_decode.h): format 0 / 1 / 2 = JSON / JSONL / YAML (write_blutils_output.rs),
// 3 = the build-tabular TSV; path NULL = stdout.  sorted: the records in query-id order, as blu_result_sort_by_query leaves them.
// two_parts: the records split into two parts that share the bean, accession and string arrays, as a multi-device result
// (the second half first unless sorted).
extern "C" int blu_sim_run_write(const int64_t* taxids, const uint64_t* off, const char* blob, uint64_t n, int taxon, int has_custom,
                                 const int32_t* custom8, int strategy, const char* text, uint64_t nbytes, const char* headers_nl, uint64_t headers_len,
                                 int sorted, int two_parts, const char* out_path, int format, const char* run_id, char* err, int errlen) {
    int wrc = 0;
    auto write = [&](const ResultView& v0) {
        ResultView v = v0;
        const ResultPart& p = v0.parts[0];
        std::vector<blu_record> recs(p.rec, p.rec + p.n_rec);
        if (sorted) {
            std::stable_sort(recs.begin(), recs.end(), [&](const blu_record& a, const blu_record& b) { return rec_query(p, a) < rec_query(p, b); });
            v.sorted = true;
        }
        ResultPart lo = p, hi = p;
        lo.rec = recs.data();
        if (two_parts) {
            lo.n_rec = p.n_rec / 2;
            hi.rec = recs.data() + lo.n_rec;
            hi.n_rec = p.n_rec - lo.n_rec;
            v.parts = sorted ? std::vector<ResultPart>{lo, hi} : std::vector<ResultPart>{hi, lo};
        } else
            v.parts = {lo};
        wrc = format == 3 ? view_write_tabular(&v, out_path, run_id) : view_write(&v, out_path, format, run_id);
    };
    const int rc = sim_run_impl(taxids, off, blob, n, taxon, has_custom, custom8, strategy, text, nbytes, headers_nl, headers_len, write, err, errlen);
    if (rc == BLU_OK && wrc != 0) {
        snprintf(err, errlen, "writer failed (%d)", wrc);
        return wrc;
    }
    return rc;
}

extern "C" void blu_sim_free(char* p) { free(p); }

// the product's serde_yaml string-scalar emitter (blu_decode.h yaml_str)
extern "C" int blu_sim_yaml_str(const char* s, uint64_t n, char* out, int cap) {
    std::string o;
    yaml_str(o, std::string_view(s, (size_t)n));
    if ((int)o.size() + 1 > cap) return -1;
    memcpy(out, o.data(), o.size());
    out[o.size()] = 0;
    return (int)o.size();
}

// interpolation of the product's taxonomy encoder, for the KAT vectors
extern "C" int blu_sim_interpolate(const char* ranks_nl, int taxon, int has_custom, const int32_t* custom8, double* out, int cap) {
    try {
        Cutoffs cut;
        cut.taxon = taxon;
        cut.has_custom = has_custom != 0;
        if (has_custom)
            for (int i = 0; i < 8; i++) cut.custom[i] = custom8[i];
        auto bb = make_backbone(cut);
        std::vector<RankInfo> rk;
        std::string s(ranks_nl);
        size_t pos = 0;
        while (true) {
            size_t k = s.find('\n', pos);
            rk.push_back(rank_from_str(s.substr(pos, k == std::string::npos ? std::string::npos : k - pos)));
            if (k == std::string::npos) break;
            pos = k + 1;
        }
        std::vector<const RankInfo*> ptr;
        for (auto& r : rk) ptr.push_back(&r);
        auto v = interpolate_cutoffs(ptr, bb);
        if ((int)v.size() > cap) return -1;
        for (size_t i = 0; i < v.size(); i++) out[i] = v[i];
        return (int)v.size();
    } catch (...) {
        return -2;
    }
}

// custom cutoff file parser of the product
extern "C" int blu_sim_custom_cutoffs(const char* path, int32_t* out8, char* err, int errlen) {
    try {
        Cutoffs c;
        read_custom_cutoffs(path, c);
        for (int i = 0; i < 8; i++) out8[i] = c.custom[i];
        return 0;
    } catch (const std::exception& e) {
        snprintf(err, errlen, "%s", e.what());
        return 2;
    }
}

// taxonomy JSON reader of the product: returns number of taxa, or -1 (I/O class error)
extern "C" long long blu_sim_read_taxonomy_json(const char* path, int use_taxid, char* err, int errlen) {
    try {
        std::vector<int64_t> ids;
        std::vector<uint64_t> off;
        std::string blob;
        read_taxonomy_json(path, use_taxid != 0, ids, off, blob);
        return (long long)ids.size();
    } catch (const std::exception& e) {
        snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// What the product's reader took from a `.blutils.json`: "taxid\0lineage\0" for every taxon, in file order (malloc'ed; the
// lineage is the text or the numeric one, as build_consensus_identities/mod.rs:287-291 chooses by use_taxid).
extern "C" int blu_sim_dump_taxonomy_json(const char* path, int use_taxid, char** out, uint64_t* out_len, char* err, int errlen) {
    try {
        std::vector<int64_t> ids;
        std::vector<uint64_t> off;
        std::string blob;
        read_taxonomy_json(path, use_taxid != 0, ids, off, blob);
        std::string o;
        for (size_t i = 0; i < ids.size(); i++) {
            o += std::to_string(ids[i]);
            o.push_back('\0');
            o.append(blob, off[i], off[i + 1] - off[i]);
            o.push_back('\0');
        }
        *out = (char*)malloc(o.size() + 1);
        memcpy(*out, o.data(), o.size());
        *out_len = o.size();
        return 0;
    } catch (const std::exception& e) {
        snprintf(err, errlen, "%s", e.what());
        return 1;
    }
}

// Side-car taxonomy cache of the product (same sequence as blu_taxonomy_load_json_cached, minus the upload):
// *state = 1 loaded from the cache, 0 built + written, -1 built, not writable.  *checksum covers every field of the
// resulting HostTaxonomy, so "loaded" and "built" can be compared.
extern "C" int blu_sim_taxonomy_cached(const char* json_path, const char* cache_path, int use_taxid, int taxon, int has_custom, const int32_t* custom8,
                                       int* state, uint64_t* checksum, char* err, int errlen) {
    try {
        Cutoffs cut;
        cut.taxon = taxon;
        cut.has_custom = has_custom != 0;
        if (has_custom)
            for (int i = 0; i < 8; i++) cut.custom[i] = custom8[i];
        const TaxCacheKey key = make_cache_key(json_path, use_taxid != 0, cut);
        HostTaxonomy T;
        *state = 1;
        if (!load_taxonomy_cache(cache_path, key, T)) {
            std::vector<int64_t> ids;
            std::vector<uint64_t> off;
            std::string blob;
            read_taxonomy_json(json_path, use_taxid != 0, ids, off, blob);
            static const uint64_t zero = 0;
            build_taxonomy(ids.data(), ids.empty() ? &zero : off.data(), blob.data(), ids.size(), cut, T);
            *state = 0;
            try {
                save_taxonomy_cache(cache_path, key, T);
            } catch (const IoErr&) {
                *state = -1;
            }
        }
        uint64_t h = 1469598103934665603ull;
        auto mixin = [&](const void* p, size_t n) {
            const unsigned char* b = (const unsigned char*)p;
            for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
            h = (h ^ n) * 1099511628211ull;
        };
        auto vec = [&](const auto& v) { mixin(v.data(), v.size() * sizeof(v[0])); };
        for (const RankInfo& r : T.ranks) {
            mixin(&r.def, sizeof r.def);
            mixin(r.slug.data(), r.slug.size()), mixin(r.display.data(), r.display.size()), mixin(r.full.data(), r.full.size());
        }
        for (const std::string& s : T.idents) mixin(s.data(), s.size());
        vec(T.taxids), vec(T.lin_off), vec(T.lin_ok), vec(T.pos_rank), vec(T.pos_ident), vec(T.lvl_key), vec(T.bean_key), vec(T.ident_rank);
        vec(T.cut), vec(T.rank_cls), vec(T.allowed_cls);
        for (const HashSlot& s : T.slots) mixin(&s.key, 8), mixin(&s.val, 4), mixin(&s.used, 4);
        mixin(&T.hash_mask, 4);
        *checksum = h;
        return 0;
    } catch (const IoErr& e) {
        snprintf(err, errlen, "%s", e.what());
        return 1;
    } catch (const std::exception& e) {
        snprintf(err, errlen, "%s", e.what());
        return 2;
    }
}
