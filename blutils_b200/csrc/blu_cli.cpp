// blu_cli.cpp -- `blu blastn build-consensus` and `blu blastn build-tabular` shims over the C ABI.
// Argument surface = BuildConsensusArguments (reference ports/cli/src/cmds/blast/commands.rs:105-143) plus the
// global flags of CliLauncher (ports/cli/src/models/cli_launcher.rs:7-22), which this stage accepts and ignores
// (`--threads` never reaches the consensus stage in the reference either: cmds/blast/mod.rs:104).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/blu_consensus.h"

static void usage() {
    fprintf(stderr,
            "Usage: blu [--log-level L] [--log-file F] [--log-format F] [-t|--threads N] blastn build-consensus <BLAST_OUT>\n"
            "           -t|--tax-file <FILE> --taxon <fungi|bacteria|eukaryotes|custom> --strategy <cautious|relaxed>\n"
            "           [-c|--custom-taxon-cutoff-file <FILE>] [-u|--use-taxid] [--blutils-out-file <FILE>]\n"
            "           [--out-format <json|jsonl|yaml>] [--device N | --devices N,M,...]\n"
            "       blu blastn build-tabular [BLU_RESULT|-] [-o|--output-file <FILE>] [-i|--input-format <json|jsonl|yaml>]\n");
}

[[noreturn]] static void die(const std::string& m) {
    // the reference panics on every failure of this command (cmds/blast/mod.rs:114-116,133-135,143-145)
    fprintf(stderr, "thread 'main' panicked: %s\n", m.c_str());
    exit(101);
}

int main(int argc, char** argv) {
    std::vector<std::string> a(argv + 1, argv + argc);
    size_t i = 0;
    // global flags
    while (i < a.size() && a[i] != "blastn") {
        if (a[i] == "--log-level" || a[i] == "--log-file" || a[i] == "--log-format" || a[i] == "-t" || a[i] == "--threads")
            i += 2;
        else if (a[i] == "-h" || a[i] == "--help") {
            usage();
            return 0;
        } else {
            usage();
            return 2;
        }
    }
    if (i + 1 < a.size() && a[i] == "blastn" && a[i + 1] == "build-tabular") {
        // BuildTabularArguments (ports/cli/src/cmds/blast/commands.rs:145-161); no GPU involved
        std::string in = "-", out, fmt = "json";
        bool have_out = false, have_in = false;
        for (i += 2; i < a.size(); i++) {
            auto value = [&](const char* shortf, const char* longf, std::string& dst) {
                const std::string eq = std::string(longf) + "=";
                if (a[i] == shortf || a[i] == longf) {
                    if (i + 1 >= a.size()) die(std::string("a value is required for '") + longf + "'");
                    dst = a[++i];
                    return true;
                }
                if (a[i].rfind(eq, 0) == 0) {
                    dst = a[i].substr(eq.size());
                    return true;
                }
                return false;
            };
            if (value("-o", "--output-file", out)) {
                have_out = true;
                continue;
            }
            if (value("-i", "--input-format", fmt)) continue;
            if (a[i] != "-" && !a[i].empty() && a[i][0] == '-') {
                fprintf(stderr, "error: unexpected argument '%s'\n", a[i].c_str());
                usage();
                return 2;
            }
            if (have_in) {
                fprintf(stderr, "error: unexpected argument '%s'\n", a[i].c_str());
                return 2;
            }
            in = a[i], have_in = true;
        }
        const int format = fmt == "json" ? BLU_FORMAT_JSON : fmt == "jsonl" ? BLU_FORMAT_JSONL : fmt == "yaml" ? BLU_FORMAT_YAML : -1;
        if (format < 0) {
            fprintf(stderr, "error: invalid value '%s' for '--input-format <INPUT_FORMAT>' [possible values: json, jsonl, yaml]\n", fmt.c_str());
            return 2;
        }
        char err[1024] = {0};
        if (blu_result_file_to_tabular(in.c_str(), have_out ? out.c_str() : nullptr, format, nullptr, err, sizeof err) != BLU_OK) die(err);
        return 0;
    }
    if (i + 1 >= a.size() || a[i] != "blastn" || a[i + 1] != "build-consensus") {
        fprintf(stderr, "only `blastn build-consensus` and `blastn build-tabular` are provided by this build (the consensus-identity hot path)\n");
        usage();
        return 2;
    }
    i += 2;
    std::string blast_out, tax_file, out_file, taxon, strategy, custom_file, fmt = "json";
    bool use_taxid = false, have_out = false;
    int device = 0;
    std::vector<int> devices;  // --devices 0,1,...: the table is sharded by query range over these GPUs (one result)
    for (; i < a.size(); i++) {
        auto need = [&](const char* f) -> std::string {
            if (i + 1 >= a.size()) die(std::string("a value is required for '") + f + "'");
            return a[++i];
        };
        auto val = [&](const std::string& flag, std::string& dst) {
            if (a[i] == flag) {
                dst = need(flag.c_str());
                return true;
            }
            if (a[i].rfind(flag + "=", 0) == 0) {
                dst = a[i].substr(flag.size() + 1);
                return true;
            }
            return false;
        };
        std::string tmp;
        if (val("--tax-file", tax_file) || (a[i] == "-t" && (tax_file = need("-t"), true))) continue;
        if (val("--blutils-out-file", out_file)) {
            have_out = true;
            continue;
        }
        if (val("--taxon", taxon) || val("--strategy", strategy) || val("--out-format", fmt)) continue;
        if (val("--custom-taxon-cutoff-file", custom_file) || (a[i] == "-c" && (custom_file = need("-c"), true))) continue;
        if (val("--devices", tmp)) {
            for (size_t k = 0; k < tmp.size();) {
                size_t e = tmp.find(',', k);
                if (e == std::string::npos) e = tmp.size();
                if (e > k) devices.push_back(atoi(tmp.substr(k, e - k).c_str()));
                k = e + 1;
            }
            if (devices.empty()) die("--devices needs a comma-separated list of CUDA device ordinals");
            continue;
        }
        if (val("--device", tmp)) {
            device = atoi(tmp.c_str());
            continue;
        }
        if (a[i] == "-u" || a[i] == "--use-taxid") {
            use_taxid = true;
            continue;
        }
        if (a[i] == "--use-taxid=true" || a[i] == "--use-taxid=false") {
            use_taxid = a[i].back() == 'e' && a[i][a[i].size() - 2] == 'u';
            continue;
        }
        if (!a[i].empty() && a[i][0] == '-') {
            fprintf(stderr, "error: unexpected argument '%s'\n", a[i].c_str());
            usage();
            return 2;
        }
        if (!blast_out.empty()) {
            fprintf(stderr, "error: unexpected argument '%s'\n", a[i].c_str());
            return 2;
        }
        blast_out = a[i];
    }
    if (blast_out.empty() || tax_file.empty() || taxon.empty() || strategy.empty()) {
        usage();
        return 2;
    }
    blu_opts o;
    memset(&o, 0, sizeof o);
    o.device = device;
    if (taxon == "fungi")
        o.taxon = BLU_TAXON_FUNGI;
    else if (taxon == "bacteria")
        o.taxon = BLU_TAXON_BACTERIA;
    else if (taxon == "eukaryotes")
        o.taxon = BLU_TAXON_EUKARYOTES;
    else if (taxon == "custom")
        o.taxon = BLU_TAXON_CUSTOM;
    else {
        fprintf(stderr, "error: invalid value '%s' for '--taxon <TAXON>' [possible values: fungi, bacteria, eukaryotes, custom]\n", taxon.c_str());
        return 2;
    }
    if (strategy == "cautious")
        o.strategy = BLU_STRATEGY_CAUTIOUS;
    else if (strategy == "relaxed")
        o.strategy = BLU_STRATEGY_RELAXED;
    else {
        fprintf(stderr, "error: invalid value '%s' for '--strategy <STRATEGY>' [possible values: cautious, relaxed]\n", strategy.c_str());
        return 2;
    }
    int format = fmt == "json" ? BLU_FORMAT_JSON : fmt == "jsonl" ? BLU_FORMAT_JSONL : fmt == "yaml" ? BLU_FORMAT_YAML : -1;
    if (format < 0) {
        fprintf(stderr, "error: invalid value '%s' for '--out-format <OUT_FORMAT>' [possible values: json, jsonl, yaml]\n", fmt.c_str());
        return 2;
    }
    o.use_taxid = use_taxid;
    if (!custom_file.empty()) {
        char err[512] = {0};
        if (blu_custom_cutoffs_from_file(custom_file.c_str(), &o, err, sizeof err) != BLU_OK) die(err);
    } else if (o.taxon == BLU_TAXON_CUSTOM)
        die("Custom taxon values are required when the custom taxon option is selected.");
    blu_ctx* ctx = nullptr;
    if ((devices.empty() ? blu_ctx_create(&o, &ctx) : blu_ctx_create_multi(&o, devices.data(), (int)devices.size(), &ctx)) != BLU_OK)
        die(blu_last_error(nullptr));
    // BLU_TAX_CACHE=1: binary side-car cache next to the taxonomy file; BLU_TAX_CACHE=<path>: that file.  An
    // environment variable, not a flag: the argument list stays the reference's (commands.rs:105-143).
    const char* tc = getenv("BLU_TAX_CACHE");
    if (tc && *tc && strcmp(tc, "0") != 0) {
        if (blu_taxonomy_load_json_cached(ctx, tax_file.c_str(), strcmp(tc, "1") == 0 ? nullptr : tc, nullptr) != BLU_OK) die(blu_last_error(ctx));
    } else if (blu_taxonomy_load_json(ctx, tax_file.c_str()) != BLU_OK)
        die(blu_last_error(ctx));
    blu_result* res = nullptr;
    if (blu_consensus_run_file(ctx, blast_out.c_str(), &res) != BLU_OK) die(std::string("Unexpected error on parse blast results: ") + blu_last_error(ctx));
    // The writer's sort by query id, on the GPU from 10^7 records on (the writer then only merges the hit-less headers in).
    // A host result's ids are packed, sorted on the GPU and its records permuted on the host: on a B200 (1000 W) sort + JSONL /
    // JSON write against the writer's own host sort, q%09d ids: 1.52 / 2.31 vs 1.00 / 1.14 ms at 10^3, 139 / 226 vs 123 / 176 ms
    // at 10^6, 1360 / 1957 vs 1518 / 1807 ms at 10^7; 40-byte read names: 205 / 229 vs 188 / 214 ms at 10^6, 2081 / 2010 vs
    // 2046 / 2154 ms at 10^7 (tools/sort_scale.py, DESIGN section 9).  Below 10^7 the host sort wins; at 10^7 they are even.
    constexpr uint64_t kGpuSortMinRecords = 10000000;
    if (blu_result_num_records(res) >= kGpuSortMinRecords && blu_result_sort_by_query(ctx, res) != BLU_OK)
        die(std::string("Unexpected error on sort results: ") + blu_last_error(ctx));
    if (blu_result_write(res, have_out ? out_file.c_str() : nullptr, format, nullptr) != BLU_OK) die("Error on persist output results");
    blu_result_free(res);
    blu_ctx_destroy(ctx);
    return 0;
}
