// `sufr-b200 create`: command-line mirror of `sufr create` (reference: sufr/src/lib.rs:83-125 flag
// definitions, :321-371 create(), sufr/src/main.rs:8-41 global flags and error exit).
// `sufr-b200 count` / `sufr-b200 locate`: the reference's query commands (sufr/src/lib.rs:467-530) over a `.sufr` file
// opened into GPU memory (sufr_b200_index_open / _locate / _hits).  extract, list and summarize stay with the reference.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cerrno>
#include <cstring>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "../../include/sufr_b200.h"

namespace {

struct CreateArgs {  // sufr/src/lib.rs:85-125
    std::string input;
    uint64_t num_partitions = 16;
    bool has_mql = false;
    uint64_t max_query_len = 0;
    std::string output;
    bool has_output = false;
    bool is_dna = false, allow_ambiguity = false, ignore_softmask = false;
    char sequence_delimiter = '%';
    std::string seed_mask;
    bool has_mask = false;
    uint64_t random_seed = 42;
    // global flags (sufr/src/lib.rs:35-45); threads is accepted and unused on the GPU path
    int threads = 0;
    std::string log_level;
    std::string log_file;
    std::vector<int> devices{0};
    uint32_t index_bits = 0;  // 0 = the reference's dispatch (u32 below u32::MAX bytes, suffix_array.rs:460-470)
};

const char* g_usage = "sufr-b200 create [OPTIONS] <INPUT>";

[[noreturn]] void usage_error(const std::string& msg) {
    fprintf(stderr, "error: %s\n\nUsage: %s\n\nFor more information, try '--help'.\n", msg.c_str(), g_usage);
    exit(2);  // clap's usage-error exit code
}

// top_level: `sufr-b200` alone or `sufr-b200 --help`: the subcommands first, then the help of `create`
void print_help(bool top_level) {
    if (top_level)
        puts("Usage: sufr-b200 [-t THREADS] [-l LOG] [--log-file FILE] <COMMAND> ...\n\n"
             "Commands:\n"
             "  create  Create sufr file (alias: cr)\n"
             "  count   Count occurrences of sequences in a sufr file (see `sufr-b200 count --help`)\n"
             "  locate  Locate sequences in a sufr file (see `sufr-b200 locate --help`)\n");
    puts("Create sufr file\n\n"
         "Usage: sufr-b200 [-t THREADS] [-l LOG] [--log-file FILE] create [OPTIONS] <INPUT>\n\n"
         "Arguments:\n  <INPUT>  Input file\n\nOptions:\n"
         "  -n, --num-partitions <NUM_PARTS>   Subproblem count [default: 16]\n"
         "  -m, --max-query-len <CONTEXT>      Max context\n"
         "  -o, --output <OUTPUT>              Output file\n"
         "  -d, --dna                          Input is DNA\n"
         "  -a, --allow-ambiguity              Allow suffixes starting with ambiguity codes\n"
         "  -i, --ignore-softmask              Ignore suffixes in soft-mask/lowercase regions\n"
         "  -D, --sequence-delimiter <DELIM>   Character to separate sequences [default: %]\n"
         "  -s, --seed-mask <MASK>             Spaced seeds mask\n"
         "  -r, --random-seed <RANDSEED>       Random seed [default: 42]\n"
         "      --device <ORDINAL>             CUDA device [default: 0]\n"
         "      --devices <LIST>               CUDA devices that share the build, e.g. 0-7 or 0,2,5 (one key-range shard each)\n"
         "      --index-bits <32|64>           Width of the SA / LCP entries [default: as the reference: 32 below 4 Gi bytes]\n"
         "  -h, --help                         Print help");
}

uint64_t parse_u64(const std::string& flag, const char* v) {
    char* end = nullptr;
    if (!v || !*v || *v == '-') usage_error("invalid value '" + std::string(v ? v : "") + "' for '" + flag + "'");
    unsigned long long x = strtoull(v, &end, 10);
    if (*end) usage_error("invalid value '" + std::string(v) + "' for '" + flag + "'");
    return x;
}

std::string file_stem(const std::string& path) {  // PathBuf::file_stem (sufr/src/lib.rs:334-340)
    size_t slash = path.find_last_of('/');
    std::string base = slash == std::string::npos ? path : path.substr(slash + 1);
    if (base.empty()) return "out";
    size_t dot = base.find_last_of('.');
    if (dot == std::string::npos || dot == 0) return base;
    return base.substr(0, dot);
}

std::vector<int> parse_devices(const std::string& flag, const char* v) {  // "0-7", "0,2,5", "3"
    std::vector<int> out;
    std::string s = v ? v : "";
    size_t i = 0;
    while (i <= s.size()) {
        size_t j = s.find(',', i);
        if (j == std::string::npos) j = s.size();
        std::string part = s.substr(i, j - i);
        size_t dash = part.find('-');
        if (part.empty()) usage_error("invalid value '" + s + "' for '" + flag + "'");
        if (dash == std::string::npos) {
            out.push_back((int)parse_u64(flag, part.c_str()));
        } else {
            int lo = (int)parse_u64(flag, part.substr(0, dash).c_str()), hi = (int)parse_u64(flag, part.substr(dash + 1).c_str());
            if (hi < lo || hi - lo > 63) usage_error("invalid value '" + s + "' for '" + flag + "'");
            for (int d = lo; d <= hi; d++) out.push_back(d);
        }
        i = j + 1;
    }
    return out;
}

double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

// ------------------------------------------------------------------ count / locate
void print_query_help(bool locate) {
    if (locate)
        puts("Locate sequences\n\n"
             "Usage: sufr-b200 locate [OPTIONS] <SUFR> [QUERY]...\n\n"
             "Arguments:\n  <SUFR>      Sufr file\n  [QUERY]...  Query strings\n\nOptions:\n"
             "  -f, --query-file <FILE>       Read queries from a file, one per line (empty lines are skipped)\n"
             "  -m, --max-query-len <LEN>     Maximum query length: only the first LEN symbols (seed-mask positions) must match\n"
             "  -a, --abs                     Show absolute position in the text: one line `QUERY POS POS ...`, in suffix order\n"
             "      --low-memory              Search the full suffix array (default: the LCP-subsampled array when\n"
             "                                --max-query-len is shorter than the one the file was built with)\n"
             "      --device <ORDINAL>        CUDA device [default: 0]\n"
             "  -h, --help                    Print help\n\n"
             "Output: per query the query line, then one line `NAME POS,POS,...` per sequence that holds a match (names in\n"
             "byte order, positions ascending), then `//`.  A query without a match prints its line and `//` only\n"
             "(with --abs: the query alone on its line).");
    else
        puts("Count occurrences of sequences\n\n"
             "Usage: sufr-b200 count [OPTIONS] <SUFR> [QUERY]...\n\n"
             "Arguments:\n  <SUFR>      Sufr file\n  [QUERY]...  Query strings\n\nOptions:\n"
             "  -f, --query-file <FILE>       Read queries from a file, one per line (empty lines are skipped)\n"
             "  -m, --max-query-len <LEN>     Maximum query length: only the first LEN symbols (seed-mask positions) must match\n"
             "      --low-memory              Search the full suffix array (default: the LCP-subsampled array when\n"
             "                                --max-query-len is shorter than the one the file was built with)\n"
             "      --device <ORDINAL>        CUDA device [default: 0]\n"
             "  -h, --help                    Print help\n\n"
             "Output: one line `QUERY COUNT` per query, in the order given (COUNT is 0 for a query without a match).");
}

struct Out {  // buffered stdout: a locate of frequent queries prints millions of positions
    std::string buf;
    void put(const std::string& s) { buf += s; flush_if(); }
    void put(const char* p, size_t n) { buf.append(p, n); flush_if(); }
    void num(uint64_t v) {
        char t[24];
        int k = snprintf(t, sizeof(t), "%llu", (unsigned long long)v);
        buf.append(t, (size_t)k);
    }
    void flush_if() { if (buf.size() > (1u << 20)) flush(); }
    void flush() { fwrite(buf.data(), 1, buf.size(), stdout); buf.clear(); }
};

int run_query(int argc, char** argv, bool locate) {
    g_usage = locate ? "sufr-b200 locate [OPTIONS] <SUFR> [QUERY]..." : "sufr-b200 count [OPTIONS] <SUFR> [QUERY]...";
    bool has_mql = false, low_memory = false, abs = false;
    uint64_t mql = 0;
    int device = 0;
    std::vector<std::string> pos, files;
    bool saw_cmd = false;
    for (int i = 1; i < argc; i++) {
        std::string s = argv[i];
        auto value = [&](const std::string& flag) -> const char* {
            size_t eq = s.find('=');
            if (s.rfind("--", 0) == 0 && eq != std::string::npos) return argv[i] + eq + 1;
            if (i + 1 >= argc) usage_error("a value is required for '" + flag + "' but none was supplied");
            return argv[++i];
        };
        std::string key = s.rfind("--", 0) == 0 ? s.substr(0, s.find('=')) : s;
        if (key == "-h" || key == "--help") { print_query_help(locate); return 0; }
        else if (key == "-t" || key == "--threads") parse_u64(key, value(key));  // global flags: accepted, unused
        else if (key == "-l" || key == "--log" || key == "--log-file") value(key);
        else if (key == "-m" || key == "--max-query-len") { mql = parse_u64(key, value(key)); has_mql = true; }
        else if (key == "--low-memory") low_memory = true;
        else if (key == "--device") device = (int)parse_u64(key, value(key));
        else if (key == "-f" || key == "--query-file") files.push_back(value(key));
        else if (locate && (key == "-a" || key == "--abs")) abs = true;
        else if (!s.empty() && s[0] == '-' && s.size() > 1) usage_error("unexpected argument '" + s + "' found");
        else if (!saw_cmd && s == (locate ? "locate" : "count")) saw_cmd = true;
        else pos.push_back(s);
    }
    if (pos.empty()) usage_error("the following required arguments were not provided:\n  <SUFR>");
    const std::string path = pos[0];
    std::vector<std::string> queries(pos.begin() + 1, pos.end());
    for (const auto& f : files) {
        FILE* fp = fopen(f.c_str(), "rb");
        if (!fp) { fprintf(stderr, "Error: %s: %s\n", f.c_str(), strerror(errno)); return 1; }
        std::string line;
        int c;
        auto push = [&] {
            if (!line.empty() && line.back() == '\r') line.pop_back();
            if (!line.empty()) queries.push_back(line);
            line.clear();
        };
        while ((c = fgetc(fp)) != EOF) {
            if (c == '\n') push(); else line.push_back((char)c);
        }
        push();
        fclose(fp);
    }
    if (queries.empty()) usage_error("the following required arguments were not provided:\n  <QUERY>...");

    SufrB200FileInfo info;
    if (sufr_b200_file_info(path.c_str(), &info) != SUFR_B200_OK) {
        fprintf(stderr, "Error: %s\n", sufr_b200_last_error());
        return 1;
    }
    SufrB200Ctx* ctx = nullptr;
    SufrB200Index* idx = nullptr;
    auto fail = [&]() {
        fprintf(stderr, "Error: %s\n", sufr_b200_last_error());
        if (idx) sufr_b200_index_free(idx);
        if (ctx) sufr_b200_ctx_destroy(ctx);
        sufr_b200_file_info_free(&info);
        return 1;
    };
    if (sufr_b200_ctx_create(device, &ctx) != SUFR_B200_OK) return fail();
    if (sufr_b200_index_open(ctx, path.c_str(), &idx) != SUFR_B200_OK) return fail();

    const uint64_t nq = queries.size();
    std::string blob;
    std::vector<uint64_t> offsets(nq + 1, 0);
    for (uint64_t i = 0; i < nq; i++) {
        blob += queries[i];
        offsets[i + 1] = blob.size();
    }
    std::vector<uint64_t> rb(nq), re(nq), ho(nq + 1);
    if (sufr_b200_index_locate(idx, (const uint8_t*)blob.data(), offsets.data(), nq, has_mql, mql, low_memory, rb.data(),
                               re.data(), ho.data()) != SUFR_B200_OK)
        return fail();

    Out out;
    if (!locate) {
        for (uint64_t i = 0; i < nq; i++) {
            out.put(queries[i]);
            out.put(" ", 1);
            out.num(ho[i + 1] - ho[i]);
            out.put("\n", 1);
        }
    } else {
        // names in byte order: rank of every record's name (equal names share a rank and a line)
        const uint64_t ns = info.num_sequences;
        std::vector<uint64_t> order(ns), name_rank(ns + 1);
        for (uint64_t i = 0; i < ns; i++) order[i] = i;
        std::sort(order.begin(), order.end(),
                  [&](uint64_t x, uint64_t y) { return strcmp(info.sequence_names[x], info.sequence_names[y]) < 0; });
        std::vector<const char*> rank_name;
        for (uint64_t k = 0; k < ns; k++) {
            if (k == 0 || strcmp(info.sequence_names[order[k]], info.sequence_names[order[k - 1]]) != 0)
                rank_name.push_back(info.sequence_names[order[k]]);
            name_rank[order[k]] = rank_name.size() - 1;
        }
        name_rank[ns] = rank_name.size();
        rank_name.push_back("");  // hits outside every record (an index without sequence starts)

        const uint64_t total = ho[nq], window = 1ull << 24;
        std::vector<uint64_t> suf, seq, spos;
        std::vector<std::pair<uint64_t, uint64_t>> cur;  // (name rank, position) of the current query
        uint64_t q = 0;
        auto begin_query = [&](uint64_t i) {
            out.put(queries[i]);
            if (!abs) out.put("\n", 1);
        };
        auto end_query = [&]() {
            if (abs) { out.put("\n", 1); return; }
            std::sort(cur.begin(), cur.end());
            for (size_t k = 0; k < cur.size();) {
                out.put(rank_name[cur[k].first]);
                out.put(" ", 1);
                size_t j = k;
                for (; j < cur.size() && cur[j].first == cur[k].first; j++) {
                    if (j > k) out.put(",", 1);
                    out.num(cur[j].second);
                }
                out.put("\n", 1);
                k = j;
            }
            out.put("//\n", 3);
            cur.clear();
        };
        while (q < nq && ho[q + 1] == 0) { begin_query(q); end_query(); q++; }
        if (q < nq) begin_query(q);
        for (uint64_t first = 0; first < total; first += window) {
            const uint64_t count = std::min(window, total - first);
            suf.resize(count);
            seq.resize(count);
            spos.resize(count);
            if (sufr_b200_index_hits(idx, first, count, suf.data(), abs ? nullptr : seq.data(), abs ? nullptr : spos.data()) !=
                SUFR_B200_OK)
                return fail();
            for (uint64_t k = 0; k < count; k++) {
                const uint64_t h = first + k;
                while (h >= ho[q + 1]) {  // the hits of query q are done: close it and every empty query behind it
                    end_query();
                    q++;
                    begin_query(q);
                }
                if (abs) {
                    out.put(" ", 1);
                    out.num(suf[k]);
                } else {
                    cur.push_back({seq[k] == UINT64_MAX ? ns : name_rank[seq[k]], spos[k]});
                }
            }
        }
        if (q < nq) {
            end_query();
            for (q++; q < nq; q++) { begin_query(q); end_query(); }
        }
    }
    out.flush();
    sufr_b200_index_free(idx);
    sufr_b200_ctx_destroy(ctx);
    sufr_b200_file_info_free(&info);
    return 0;
}

int main(int argc, char** argv) {
    // the subcommand is the first of the known names on the command line
    for (int i = 1; i < argc; i++) {
        const std::string s = argv[i];
        if (s == "create" || s == "cr") break;
        if (s == "count" || s == "locate") return run_query(argc, argv, s == "locate");
    }
    CreateArgs a;
    std::vector<std::string> pos;
    bool saw_create = false;
    for (int i = 1; i < argc; i++) {
        std::string s = argv[i];
        auto value = [&](const std::string& flag) -> const char* {
            size_t eq = s.find('=');
            if (s.rfind("--", 0) == 0 && eq != std::string::npos) return argv[i] + eq + 1;
            if (i + 1 >= argc) usage_error("a value is required for '" + flag + "' but none was supplied");
            return argv[++i];
        };
        std::string key = s.rfind("--", 0) == 0 ? s.substr(0, s.find('=')) : s;
        if (key == "-h" || key == "--help") { print_help(!saw_create); return 0; }
        else if (key == "-t" || key == "--threads") a.threads = (int)parse_u64(key, value(key));
        else if (key == "-l" || key == "--log") a.log_level = value(key);
        else if (key == "--log-file") a.log_file = value(key);
        else if (key == "-n" || key == "--num-partitions") a.num_partitions = parse_u64(key, value(key));
        else if (key == "-m" || key == "--max-query-len") { a.max_query_len = parse_u64(key, value(key)); a.has_mql = true; }
        else if (key == "-o" || key == "--output") { a.output = value(key); a.has_output = true; }
        else if (key == "-d" || key == "--dna") a.is_dna = true;
        else if (key == "-a" || key == "--allow-ambiguity") a.allow_ambiguity = true;
        else if (key == "-i" || key == "--ignore-softmask") a.ignore_softmask = true;
        else if (key == "-D" || key == "--sequence-delimiter") {
            const char* v = value(key);
            if (strlen(v) != 1) usage_error("invalid value '" + std::string(v) + "' for '--sequence-delimiter <DELIM>'");
            a.sequence_delimiter = v[0];
        }
        else if (key == "-s" || key == "--seed-mask") { a.seed_mask = value(key); a.has_mask = true; }
        else if (key == "-r" || key == "--random-seed") a.random_seed = parse_u64(key, value(key));
        else if (key == "--device") a.devices = {(int)parse_u64(key, value(key))};
        else if (key == "--devices") a.devices = parse_devices(key, value(key));
        else if (key == "--index-bits") {
            a.index_bits = (uint32_t)parse_u64(key, value(key));
            if (a.index_bits != 32 && a.index_bits != 64) usage_error("invalid value for '--index-bits <32|64>'");
        }
        else if (!s.empty() && s[0] == '-' && s.size() > 1) usage_error("unexpected argument '" + s + "' found");
        else if (!saw_create && (s == "create" || s == "cr")) saw_create = true;
        else pos.push_back(s);
    }
    if (!saw_create) {
        if (argc <= 1) { print_help(true); return 2; }
        usage_error("unrecognized subcommand (sufr-b200 provides 'create', 'count' and 'locate')");
    }
    if (pos.size() != 1) usage_error(pos.empty() ? "the following required arguments were not provided:\n  <INPUT>"
                                                 : "unexpected argument '" + pos[1] + "' found");
    a.input = pos[0];
    if (a.has_mql && a.has_mask)  // clap conflicts_with (sufr/src/lib.rs:95)
        usage_error("the argument '--max-query-len <CONTEXT>' cannot be used with '--seed-mask <MASK>'");

    const bool info = a.log_level == "info" || a.log_level == "debug";
    FILE* logf = stdout;
    if (info && !a.log_file.empty()) {
        logf = fopen(a.log_file.c_str(), "w");
        if (!logf) { fprintf(stderr, "Error: %s: cannot open log file\n", a.log_file.c_str()); return 1; }
    }

    double t0 = now_s();
    SufrB200Sequences seqs;
    if (sufr_b200_read_sequence_file(a.input.c_str(), (uint8_t)a.sequence_delimiter, &seqs) != SUFR_B200_OK) {
        fprintf(stderr, "Error: %s\n", sufr_b200_last_error());
        return 1;
    }
    if (info) fprintf(logf, "Read input of len %llu in %.3fs\n", (unsigned long long)seqs.seq_len, now_s() - t0);

    std::string outfile = a.has_output ? a.output : file_stem(a.input) + ".sufr";
    SufrB200Args args;
    memset(&args, 0, sizeof(args));
    args.text = seqs.seq;
    args.text_len = seqs.seq_len;
    args.path = outfile.c_str();
    args.low_memory = 1;
    args.has_max_query_len = a.has_mql;
    args.max_query_len = a.max_query_len;
    args.is_dna = a.is_dna;
    args.allow_ambiguity = a.allow_ambiguity;
    args.ignore_softmask = a.ignore_softmask;
    args.sequence_starts = seqs.start_positions;
    args.sequence_names = (const char* const*)seqs.sequence_names;
    args.num_sequences = seqs.num_sequences;
    args.num_partitions = a.num_partitions;
    args.seed_mask = a.has_mask ? a.seed_mask.c_str() : nullptr;
    args.random_seed = a.random_seed;
    args.rank = 0;
    args.world_size = 1;

    t0 = now_s();
    SufrB200Result res;
    int rc = (a.devices.size() == 1 && a.index_bits == 0)
                 ? sufr_b200_create(&args, a.devices[0], &res)
                 : sufr_b200_create_multi(&args, a.devices.data(), (int)a.devices.size(), a.index_bits, &res);
    if (rc != SUFR_B200_OK) {
        fprintf(stderr, "Error: %s\n", sufr_b200_last_error());  // sufr/src/main.rs:9-12
        sufr_b200_sequences_free(&seqs);
        return 1;
    }
    if (info) {
        const SufrB200Timings& t = res.timings;
        fprintf(logf, "Encoded text (alphabet %u, %u bits/symbol) in %.3fms\n", res.alphabet_size, res.bits_per_symbol,
                t.encode_ms);
        fprintf(logf, "Sorted %llu suffixes on %zu GPU%s in %.3fms (keys %.3f, sort %.3f, refine %.3f [%u word / %u doubling rounds], "
                      "lcp %.3f, finish %.3f; h2d %.3f, d2h %.3f; %llu kernel launches)\n",
                (unsigned long long)res.num_suffixes, a.devices.size(), a.devices.size() == 1 ? "" : "s", t.total_ms, t.keys_ms, t.sort_ms, t.refine_ms, res.refine_rounds,
                res.doubling_rounds, t.lcp_ms, t.finish_ms, t.h2d_ms, t.d2h_ms, (unsigned long long)res.kernel_launches);
        struct stat sb;
        unsigned long long bytes = stat(outfile.c_str(), &sb) == 0 ? (unsigned long long)sb.st_size : 0;
        fprintf(logf, "Wrote %llu byte%s to '%s' in %.3fs\n", bytes, bytes == 1 ? "" : "s", outfile.c_str(), now_s() - t0);
    }
    sufr_b200_result_free(nullptr, &res);
    sufr_b200_sequences_free(&seqs);
    if (logf != stdout) fclose(logf);
    return 0;
}
