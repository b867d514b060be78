// blu_tabular.h -- `blu blastn build-tabular`: a blutils result file (JSON, JSONL or YAML) -> the 12-column TSV.  Host only.
// Follows parse_consensus_as_tabular (reference core/src/use_cases/parse_consensus_as_tabular/mod.rs:15-173) and the
// readers it uses (core/src/domain/dtos/file_or_stdin.rs:96-176), including their quirks:
//   * the existence check looks at `<input with its extension replaced by .json>`, whatever the format (mod.rs:24-33);
//   * a JSONL config line is recognised by the substring `isConfig`; every other non-empty line must be a result, so
//     the `null` config line that build-consensus writes makes the reference (and this) fail (file_or_stdin.rs:141-172);
//   * to a file the pieces are written without line breaks, to stdout one println! per piece (see blu_decode.h).
// Serde semantics restated: unknown fields are skipped, a duplicate field is an error, Option fields may be missing or
// null, LinnaeanRank (de)serialises to the same string (`Other(String)` is untagged, linnaean_ranks.rs:14-29), f64
// fields accept any JSON number.  YAML input goes through blu_yaml_in.h (the block-style subset serde_yaml writes; anything
// else of YAML is refused with BLU_ERR_UNSUPPORTED) with serde_yaml's scalar typing.
#pragma once
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <string>
#include <string_view>
#include <vector>

#include "../../include/blu_consensus.h"
#include "blu_decode.h"
#include "blu_json.h"
#include "blu_yaml_in.h"

namespace blu {

struct TabBean {  // ConsensusBean, consensus_result.rs:37-45
    std::string rank, identifier, taxonomy;
    bool has_taxonomy = false;
    int32_t occurrences = 0;
    std::vector<std::string> accessions;
};

struct TabTaxon {  // TaxonomyBean, taxonomy_bean.rs:5-17
    std::string reached_rank, identifier, taxonomy;
    bool has_taxonomy = false, mutated = false, single_match = false, has_beans = false;
    double perc_identity = 0, bit_score = 0;
    std::vector<TabBean> beans;
};

struct TabResult {  // QueryWithConsensus, consensus_result.rs:7-13
    std::string run_id, query;
    bool has_run_id = false, has_taxon = false;
    TabTaxon taxon;
};

namespace tabular_detail {

// PathBuf::set_extension: the extension starts at the last '.' of the file name, unless that dot begins the name
inline std::string set_extension(const char* path, const char* ext) {
    std::string p = path;
    const size_t slash = p.find_last_of('/');
    const size_t dot = p.find_last_of('.');
    if (dot != std::string::npos && dot > (slash == std::string::npos ? 0 : slash + 1)) p.resize(dot);
    return p + ext;
}

// uuid::Uuid from a string (hyphenated, simple, braced or urn form) -> its Display form (hyphenated, lower case)
inline std::string parse_uuid(JsonCursor& c, const std::string& s) {
    std::string_view v(s);
    if (v.size() >= 9 && (v.substr(0, 9) == "urn:uuid:")) v.remove_prefix(9);
    if (v.size() >= 2 && v.front() == '{' && v.back() == '}') v = v.substr(1, v.size() - 2);
    std::string hex;
    if (v.size() == 36) {
        for (size_t i = 0; i < 36; i++) {
            const bool dash = i == 8 || i == 13 || i == 18 || i == 23;
            if (dash != (v[i] == '-')) c.fail("invalid UUID");
            if (!dash) hex.push_back(v[i]);
        }
    } else
        hex.assign(v);
    if (hex.size() != 32) c.fail("invalid UUID");
    std::string out;
    for (size_t i = 0; i < 32; i++) {
        char ch = hex[i];
        if (ch >= 'A' && ch <= 'F') ch = (char)(ch + 32);
        if (!((ch >= '0' && ch <= '9') || (ch >= 'a' && ch <= 'f'))) c.fail("invalid UUID");
        if (i == 8 || i == 12 || i == 16 || i == 20) out.push_back('-');
        out.push_back(ch);
    }
    return out;
}

inline double parse_f64(JsonCursor& c) {
    c.ws();
    const char* s = c.p;
    const char* q = s;
    if (q < c.e && *q == '-') q++;
    const char* d0 = q;
    while (q < c.e && *q >= '0' && *q <= '9') q++;
    if (q == d0 || (q - d0 > 1 && *d0 == '0')) c.fail("expected a number");
    if (q < c.e && *q == '.') {
        const char* f0 = ++q;
        while (q < c.e && *q >= '0' && *q <= '9') q++;
        if (q == f0) c.fail("expected a number");
    }
    if (q < c.e && (*q == 'e' || *q == 'E')) {
        q++;
        if (q < c.e && (*q == '+' || *q == '-')) q++;
        const char* x0 = q;
        while (q < c.e && *q >= '0' && *q <= '9') q++;
        if (q == x0) c.fail("expected a number");
    }
    const std::string lit(s, q);
    c.p = q;
    return strtod(lit.c_str(), nullptr);  // correctly rounded (serde_json: exact for the <= 17-digit values the writer emits)
}

inline bool parse_bool(JsonCursor& c) {
    c.ws();
    if (c.e - c.p >= 4 && !memcmp(c.p, "true", 4)) {
        c.p += 4;
        return true;
    }
    if (c.e - c.p >= 5 && !memcmp(c.p, "false", 5)) {
        c.p += 5;
        return false;
    }
    c.fail("expected a boolean");
}

inline void need_string(JsonCursor& c, std::string& out) {
    if (c.peek() != '"') c.fail("expected a string");
    out.clear();
    c.string(&out);
}

// Option<String>: string or null
inline bool opt_string(JsonCursor& c, std::string& out) {
    if (c.consume_null()) return false;
    need_string(c, out);
    return true;
}

struct Seen {
    uint32_t bits = 0;
    void once(JsonCursor& c, int i, const char* name) {
        if (bits >> i & 1) c.fail((std::string("duplicate field `") + name + "`").c_str());
        bits |= 1u << i;
    }
    void require(JsonCursor& c, int i, const char* name) const {
        if (!(bits >> i & 1)) c.fail((std::string("missing field `") + name + "`").c_str());
    }
};

inline void parse_bean(JsonCursor& c, TabBean& b) {
    Seen seen;
    std::string key;
    c.expect('{');
    if (!c.consume('}')) {
        do {
            need_string(c, key);
            c.expect(':');
            if (key == "rank")
                seen.once(c, 0, "rank"), need_string(c, b.rank);
            else if (key == "identifier")
                seen.once(c, 1, "identifier"), need_string(c, b.identifier);
            else if (key == "occurrences") {
                seen.once(c, 2, "occurrences");
                const int64_t v = c.i64();
                if (v < INT32_MIN || v > INT32_MAX) c.fail("occurrences does not fit i32");
                b.occurrences = (int32_t)v;
            } else if (key == "taxonomy")
                seen.once(c, 3, "taxonomy"), b.has_taxonomy = opt_string(c, b.taxonomy);
            else if (key == "accessions") {
                seen.once(c, 4, "accessions");
                c.expect('[');
                if (!c.consume(']')) {
                    do {
                        b.accessions.emplace_back();
                        need_string(c, b.accessions.back());
                    } while (c.consume(','));
                    c.expect(']');
                }
            } else
                c.skip_value();
        } while (c.consume(','));
        c.expect('}');
    }
    seen.require(c, 0, "rank"), seen.require(c, 1, "identifier"), seen.require(c, 2, "occurrences"), seen.require(c, 4, "accessions");
}

inline void parse_taxon(JsonCursor& c, TabTaxon& t) {
    Seen seen;
    std::string key, tmp;
    c.expect('{');
    if (!c.consume('}')) {
        do {
            need_string(c, key);
            c.expect(':');
            if (key == "reachedRank")
                seen.once(c, 0, "reachedRank"), need_string(c, t.reached_rank);
            else if (key == "maxAllowedRank") {
                seen.once(c, 1, "maxAllowedRank");
                opt_string(c, tmp);  // Option<LinnaeanRank>: not printed
            } else if (key == "identifier")
                seen.once(c, 2, "identifier"), need_string(c, t.identifier);
            else if (key == "percIdentity")
                seen.once(c, 3, "percIdentity"), t.perc_identity = parse_f64(c);
            else if (key == "bitScore")
                seen.once(c, 4, "bitScore"), t.bit_score = parse_f64(c);
            else if (key == "taxonomy")
                seen.once(c, 5, "taxonomy"), t.has_taxonomy = opt_string(c, t.taxonomy);
            else if (key == "mutated")
                seen.once(c, 6, "mutated"), t.mutated = parse_bool(c);
            else if (key == "singleMatch")
                seen.once(c, 7, "singleMatch"), t.single_match = parse_bool(c);
            else if (key == "consensusBeans") {
                seen.once(c, 8, "consensusBeans");
                if (!c.consume_null()) {
                    t.has_beans = true;
                    c.expect('[');
                    if (!c.consume(']')) {
                        do {
                            t.beans.emplace_back();
                            parse_bean(c, t.beans.back());
                        } while (c.consume(','));
                        c.expect(']');
                    }
                }
            } else
                c.skip_value();
        } while (c.consume(','));
        c.expect('}');
    }
    seen.require(c, 0, "reachedRank"), seen.require(c, 2, "identifier"), seen.require(c, 3, "percIdentity"), seen.require(c, 4, "bitScore");
    seen.require(c, 6, "mutated"), seen.require(c, 7, "singleMatch");
}

inline void parse_result(JsonCursor& c, TabResult& r) {
    if (c.peek() != '{') c.fail("invalid type, expected struct QueryWithConsensus");
    Seen seen;
    std::string key, tmp;
    c.expect('{');
    if (!c.consume('}')) {
        do {
            need_string(c, key);
            c.expect(':');
            if (key == "runId") {
                seen.once(c, 0, "runId");
                if ((r.has_run_id = opt_string(c, tmp))) r.run_id = parse_uuid(c, tmp);
            } else if (key == "query")
                seen.once(c, 1, "query"), need_string(c, r.query);
            else if (key == "taxon") {
                seen.once(c, 2, "taxon");
                if (!c.consume_null()) {
                    r.has_taxon = true;
                    parse_taxon(c, r.taxon);
                }
            } else
                c.skip_value();
        } while (c.consume(','));
        c.expect('}');
    }
    seen.require(c, 1, "query");
}

// BlastBuilder (the `config` echo of run-with-consensus): only its runId is used here (mod.rs:97-100)
inline bool parse_config_run_id(JsonCursor& c, std::string& run_id) {
    if (c.consume_null()) return false;
    bool have = false;
    std::string key, tmp;
    c.expect('{');
    if (!c.consume('}')) {
        do {
            need_string(c, key);
            c.expect(':');
            if (key == "runId") {
                need_string(c, tmp);
                run_id = parse_uuid(c, tmp);
                have = true;
            } else
                c.skip_value();
        } while (c.consume(','));
        c.expect('}');
    }
    if (!have) c.fail("missing field `runId`");
    return true;
}

// ---- the same structs from a YAML document (blu_yaml_in.h) -----------------------------------------------------------------
inline const YNode* yaml_field(const YNode& m, const char* name) {
    for (auto& kv : m.map)
        if (kv.first == name) return kv.second.get();
    return nullptr;
}
inline const YNode& yaml_need(const YNode& m, const char* name) {
    const YNode* n = yaml_field(m, name);
    if (!n) yaml_typed::bad(m, std::string("missing field `") + name + "`");
    return *n;
}
inline void yaml_need_map(const YNode& n, const char* what) {
    if (n.kind != YNode::Map) yaml_typed::bad(n, std::string("invalid type: expected struct ") + what);
}
inline bool yaml_opt_string(const YNode& m, const char* name, std::string& out) {
    const YNode* n = yaml_field(m, name);
    if (!n || yaml_typed::is_null(*n)) return false;
    out = yaml_typed::as_str(*n, name);
    return true;
}
inline std::string yaml_uuid(const YNode& n, const std::string& s) {
    JsonCursor c(s.data(), s.size());
    try {
        return parse_uuid(c, s);
    } catch (const JsonError&) {
        yaml_typed::bad(n, "invalid UUID");
    }
}

inline void yaml_bean(const YNode& n, TabBean& b) {
    yaml_need_map(n, "ConsensusBean");
    b.rank = yaml_typed::as_str(yaml_need(n, "rank"), "rank");
    b.identifier = yaml_typed::as_str(yaml_need(n, "identifier"), "identifier");
    const int64_t occ = yaml_typed::as_i64(yaml_need(n, "occurrences"), "occurrences");
    if (occ < INT32_MIN || occ > INT32_MAX) yaml_typed::bad(n, "occurrences does not fit i32");
    b.occurrences = (int32_t)occ;
    b.has_taxonomy = yaml_opt_string(n, "taxonomy", b.taxonomy);
    const YNode& acc = yaml_need(n, "accessions");
    if (acc.kind != YNode::Seq) yaml_typed::bad(acc, "invalid type: expected a sequence for accessions");
    for (auto& a : acc.seq) b.accessions.push_back(yaml_typed::as_str(*a, "accessions"));
}

inline void yaml_taxon(const YNode& n, TabTaxon& t) {
    yaml_need_map(n, "TaxonomyBean");
    t.reached_rank = yaml_typed::as_str(yaml_need(n, "reachedRank"), "reachedRank");
    std::string tmp;
    yaml_opt_string(n, "maxAllowedRank", tmp);  // Option<LinnaeanRank>: not printed
    t.identifier = yaml_typed::as_str(yaml_need(n, "identifier"), "identifier");
    t.perc_identity = yaml_typed::as_f64(yaml_need(n, "percIdentity"), "percIdentity");
    t.bit_score = yaml_typed::as_f64(yaml_need(n, "bitScore"), "bitScore");
    t.has_taxonomy = yaml_opt_string(n, "taxonomy", t.taxonomy);
    t.mutated = yaml_typed::as_bool(yaml_need(n, "mutated"), "mutated");
    t.single_match = yaml_typed::as_bool(yaml_need(n, "singleMatch"), "singleMatch");
    const YNode* beans = yaml_field(n, "consensusBeans");
    if (beans && !yaml_typed::is_null(*beans)) {
        if (beans->kind != YNode::Seq) yaml_typed::bad(*beans, "invalid type: expected a sequence for consensusBeans");
        t.has_beans = true;
        for (auto& b : beans->seq) {
            t.beans.emplace_back();
            yaml_bean(*b, t.beans.back());
        }
    }
}

inline void yaml_result(const YNode& n, TabResult& r) {
    yaml_need_map(n, "QueryWithConsensus");
    std::string tmp;
    if ((r.has_run_id = yaml_opt_string(n, "runId", tmp))) r.run_id = yaml_uuid(n, tmp);
    r.query = yaml_typed::as_str(yaml_need(n, "query"), "query");
    const YNode* t = yaml_field(n, "taxon");
    if (t && !yaml_typed::is_null(*t)) {
        r.has_taxon = true;
        yaml_taxon(*t, r.taxon);
    }
}

}  // namespace tabular_detail

// Returns BLU_OK, BLU_ERR_IO (with `err` set: the reference's Err(MappedErrors)) or BLU_ERR_UNSUPPORTED (YAML constructs outside
// the subset blu_yaml_in.h reads).
// in_path NULL or "-": stdin.  out_path NULL: stdout.  run_id_for_missing: used where neither a result nor the config
// carries a run id (NULL: a fresh UUIDv4, as the reference).
inline int result_file_to_tabular(const char* in_path, const char* out_path, int input_format, const char* run_id_for_missing, std::string& err) {
    using namespace tabular_detail;
    const bool from_stdin = !in_path || std::string_view(in_path) == "-";
    std::string buf;
    if (from_stdin)
        buf.assign(std::istreambuf_iterator<char>(std::cin), std::istreambuf_iterator<char>());
    else {
        if (!std::ifstream(set_extension(in_path, ".json")).good()) {
            err = std::string("The file `") + in_path + "` does not exist.";
            return BLU_ERR_IO;
        }
        std::ifstream f(in_path, std::ios::binary);
        if (!f) {
            err = std::string("unable to read `") + in_path + "`";
            return BLU_ERR_IO;
        }
        buf.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
    }
    std::vector<TabResult> results;
    std::string cfg_run_id;
    bool have_cfg = false;
    try {
        if (input_format == BLU_FORMAT_JSON) {
            JsonCursor c(buf.data(), buf.size());
            bool have_results = false, seen_cfg = false;
            std::string key;
            c.expect('{');
            if (!c.consume('}')) {
                do {
                    need_string(c, key);
                    c.expect(':');
                    if (key == "results") {
                        if (have_results) c.fail("duplicate field `results`");
                        have_results = true;
                        c.expect('[');
                        if (!c.consume(']')) {
                            do {
                                results.emplace_back();
                                parse_result(c, results.back());
                            } while (c.consume(','));
                            c.expect(']');
                        }
                    } else if (key == "config") {
                        if (seen_cfg) c.fail("duplicate field `config`");
                        seen_cfg = true;
                        have_cfg = parse_config_run_id(c, cfg_run_id);
                    } else
                        c.skip_value();
                } while (c.consume(','));
                c.expect('}');
            }
            c.end();
            if (!have_results) c.fail("missing field `results`");
        } else if (input_format == BLU_FORMAT_YAML) {
            YamlReader reader;  // (the results are converted one by one as they are read: no tree of the whole file)
            const std::unique_ptr<YNode> root = reader.parse(buf, "results", [&](const YNode& item) {
                results.emplace_back();
                yaml_result(item, results.back());
            });
            yaml_need_map(*root, "BlutilsOutput");
            const YNode& rs = yaml_need(*root, "results");
            if (rs.kind != YNode::Seq) yaml_typed::bad(rs, "invalid type: expected a sequence for results");
            const YNode* cfg = yaml_field(*root, "config");
            if (cfg && !yaml_typed::is_null(*cfg)) {
                yaml_need_map(*cfg, "BlastBuilder");
                const YNode& id = yaml_need(*cfg, "runId");
                cfg_run_id = yaml_uuid(id, yaml_typed::as_str(id, "runId"));
                have_cfg = true;
            }
        } else {
            size_t pos = 0;
            while (pos < buf.size()) {
                size_t nl = buf.find('\n', pos);
                if (nl == std::string::npos) nl = buf.size();
                size_t len = nl - pos;
                if (len && buf[pos + len - 1] == '\r') len--;  // BufRead::lines strips "\r\n"
                const std::string_view line(buf.data() + pos, len);
                pos = nl + 1;
                if (line.empty()) continue;
                JsonCursor c(line.data(), line.size());
                if (line.find("isConfig") != std::string_view::npos) {
                    have_cfg = parse_config_run_id(c, cfg_run_id);
                } else {
                    results.emplace_back();
                    parse_result(c, results.back());
                }
                c.end();
            }
        }
    } catch (const JsonError& e) {
        err = std::string(input_format == BLU_FORMAT_JSON ? "unable to parse content as JSON: " : "unable to parse line as JSON: ") + e.what();
        return BLU_ERR_IO;
    } catch (const YamlError& e) {
        err = std::string("unable to parse content as YAML: ") + e.what();
        return BLU_ERR_IO;
    } catch (const YamlUnsupported& e) {
        err = e.what();
        return BLU_ERR_UNSUPPORTED;
    }
    const std::string fallback = have_cfg ? cfg_run_id : (run_id_for_missing ? std::string(run_id_for_missing) : uuid_v4());

    const bool to_stdout = out_path == nullptr;
    FILE* f = stdout;
    if (out_path) {
        const std::string target = set_extension(out_path, ".tsv");  // remove an existing file, append (mod.rs:54-66)
        std::remove(target.c_str());
        f = fopen(target.c_str(), "ab");
        if (!f) {
            err = "could not create " + target;
            return BLU_ERR_IO;
        }
    }
    std::string o;
    auto piece_done = [&]() {
        tsv_end_piece(o, to_stdout);
        if (o.size() > (8u << 20)) {
            fwrite(o.data(), 1, o.size(), f);
            o.clear();
        }
    };
    auto or_null = [](bool has, const std::string& s) { return has ? std::string_view(s) : std::string_view("null"); };
    tsv_header(o);
    piece_done();
    for (const TabResult& r : results) {
        if (!r.has_taxon) {
            tsv_no_taxon(o, r.query);
            piece_done();
            continue;
        }
        const std::string& rid = r.has_run_id ? r.run_id : fallback;
        const TabTaxon& t = r.taxon;
        tsv_consensus(o, rid, r.query, t.reached_rank, t.identifier, t.perc_identity, t.bit_score, or_null(t.has_taxonomy, t.taxonomy), t.mutated, t.single_match);
        piece_done();
        for (const TabBean& b : t.beans) {
            tsv_blast_match(o, rid, r.query, b.rank, b.identifier, t.bit_score, or_null(b.has_taxonomy, b.taxonomy), b.occurrences);
            for (size_t a = 0; a < b.accessions.size(); a++) tsv_accession(o, a, b.accessions[a]);
            piece_done();
        }
    }
    fwrite(o.data(), 1, o.size(), f);
    if (out_path)
        fclose(f);
    else
        fflush(stdout);
    return BLU_OK;
}

}  // namespace blu
