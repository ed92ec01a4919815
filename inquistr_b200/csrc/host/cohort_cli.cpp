// cohort_cli.cpp -- `inquistr-b200 combine`, `inquistr-b200 outlier` (SURVEY 8f rank 3) and `inquistr-b200 assoc`.
// Host side of the reference's src/combine.rs:27-59 and src/outlier.rs:33-72 / src/main.rs:75-99,202-229
// above the C ABI of include/inqcohort.h: text in, text out; the per-row arithmetic runs on the GPU.
// A Rust panic in the reference maps to exit code 101, clap usage errors to 2. `assoc` has no counterpart in the
// reference's binary (DESIGN.md 5e): its input errors exit 1 with `inquistr-b200: <file>:<line>: ...`.
#include <sys/stat.h>
#include <zlib.h>

#include <algorithm>
#include <charconv>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../../include/inqcall.h"
#include "../../../include/inqcohort.h"

namespace inqhost {

namespace {

[[noreturn]] void cpanic(const std::string &msg)
{
    fprintf(stderr, "thread 'main' panicked: %s\n", msg.c_str());
    exit(101);
}
[[noreturn]] void cusage(const std::string &msg, const char *sub)
{
    fprintf(stderr, "error: %s\n\nUsage: inquistr-b200 %s\n\nFor more information, try '--help'.\n", msg.c_str(), sub);
    exit(2);
}
bool exists(const std::string &p) { struct stat st; return stat(p.c_str(), &st) == 0; }

// plain or gzip-compressed text, line by line (combine.rs:10-25 decides by the .gz extension,
// utils.rs:7-13 sniffs the content; gzread is transparent for both)
struct LineReader {
    gzFile f = nullptr;
    std::string buf;
    bool open(const std::string &path) { f = gzopen(path.c_str(), "rb"); if (f) gzbuffer(f, 1 << 20); return f != nullptr; }
    bool next(std::string &line)
    {
        line.clear();
        char tmp[1 << 16];
        bool any = false;
        while (gzgets(f, tmp, sizeof(tmp))) {
            any = true;
            const size_t n = strlen(tmp);
            if (n && tmp[n - 1] == '\n') {
                line.append(tmp, n - 1);
                if (!line.empty() && line.back() == '\r') line.pop_back();     // BufRead::lines strips \r\n too
                return true;
            }
            line.append(tmp, n);
        }
        return any;
    }
    ~LineReader() { if (f) gzclose(f); }
};

void split_tabs(const std::string &s, std::vector<std::string> &out)
{
    out.clear();
    size_t a = 0;
    for (;;) {
        const size_t b = s.find('\t', a);
        out.emplace_back(s, a, b == std::string::npos ? std::string::npos : b - a);
        if (b == std::string::npos) break;
        a = b + 1;
    }
}

// Rust's `str::parse::<f32>`: decimal digits / '.' / exponent with optional sign, or (case-insensitive)
// "nan", "inf", "infinity"; no surrounding whitespace
bool parse_f32(const std::string &s, float *out)
{
    if (s.empty()) return false;
    size_t i = (s[0] == '+' || s[0] == '-') ? 1 : 0;
    std::string low;
    for (size_t k = i; k < s.size(); ++k) low.push_back((char)tolower((unsigned char)s[k]));
    if (low == "nan") { *out = NAN; return true; }
    if (low == "inf" || low == "infinity") { *out = s[0] == '-' ? -INFINITY : INFINITY; return true; }
    bool digit = false;
    for (size_t k = i; k < s.size(); ++k) {
        const char c = s[k];
        if (c >= '0' && c <= '9') digit = true;
        else if (!(c == '.' || c == 'e' || c == 'E' || ((c == '+' || c == '-') && k > i && (s[k - 1] == 'e' || s[k - 1] == 'E')))) return false;
    }
    if (!digit) return false;
    char *end = nullptr;
    *out = strtof(s.c_str(), &end);
    return end && *end == '\0';
}

std::string strip_hap(std::string s)                           // outlier.rs:112 .replace("_H1", "").replace("_H2", "")
{
    for (const char *pat : {"_H1", "_H2"})
        for (size_t p; (p = s.find(pat)) != std::string::npos;) s.erase(p, 3);
    return s;
}

}  // namespace

// combine.rs:27-59
int combine_main(const std::vector<std::string> &files)
{
    if (files.empty()) cusage("the following required arguments were not provided:\n  <CALLS>...", "combine <CALLS>...");
    for (const auto &f : files)
        if (!exists(f)) cpanic("File " + f + " does not exist!");
    std::vector<LineReader> rd(files.size());
    for (size_t i = 0; i < files.size(); ++i)
        if (!rd[i].open(files[i])) cpanic("couldn't open " + files[i]);
    std::string line, other, out;
    std::vector<std::string> cols;
    while (rd[0].next(line)) {
        out = line;
        for (size_t i = 1; i < files.size(); ++i) {
            if (!rd[i].next(other)) cpanic("called `Option::unwrap()` on a `None` value (" + files[i] + " has fewer lines than " + files[0] + ")");
            split_tabs(other, cols);
            for (size_t c = 3; c < cols.size(); ++c) { out.push_back('\t'); out += cols[c]; }   // only the scores (combine.rs:50-54)
        }
        out.push_back('\n');
        fwrite(out.data(), 1, out.size(), stdout);
    }
    return 0;
}

// main.rs:75-99,202-229 + outlier.rs:33-72
int outlier_main(const std::vector<std::string> &v, int device)
{
    const char *usage = "outlier [OPTIONS] <COMBINED>";
    std::string combined, sample, subset_file, method = "zscore";
    bool has_sample = false, has_subset = false;
    uint64_t minsize = 10;
    float zscore = 3.0f;
    for (size_t i = 0; i < v.size(); ++i) {
        const std::string &a = v[i];
        auto value = [&](const char *name) -> std::string {
            if (i + 1 >= v.size()) cusage(std::string("a value is required for '") + name + "' but none was supplied", usage);
            return v[++i];
        };
        if (a == "--minsize") {
            const std::string s = value("--minsize <MINSIZE>");
            char *e = nullptr;
            minsize = strtoull(s.c_str(), &e, 10);
            if (s.empty() || *e || s[0] == '-' || minsize > 0xFFFFFFFFull) cusage("invalid value '" + s + "' for '--minsize <MINSIZE>'", usage);
        } else if (a == "-z" || a == "--zscore") {
            const std::string s = value("--zscore <ZSCORE>");
            if (!parse_f32(s, &zscore)) cusage("invalid value '" + s + "' for '--zscore <ZSCORE>'", usage);
        } else if (a == "--method") {
            method = value("--method <METHOD>");
            if (method != "zscore" && method != "dbscan") cusage("invalid value '" + method + "' for '--method <METHOD>'\n  [possible values: zscore, dbscan]", usage);
        } else if (a == "-s" || a == "--sample") { sample = value("--sample <SAMPLE>"); has_sample = true; }
        else if (a == "-S" || a == "--subset") { subset_file = value("--subset <SUBSET>"); has_subset = true; }
        else if (a == "-h" || a == "--help") {
            printf("Find outliers from TSV\n\nUsage: inquistr-b200 %s\n\nArguments:\n  <COMBINED>  combined file of calls\n\nOptions:\n"
                   "      --minsize <MINSIZE>  minimal length of expansion to be present in cohort [default: 10]\n"
                   "  -z, --zscore <ZSCORE>    zscore cutoff to decide if a value is an outlier [default: 3]\n"
                   "      --method <METHOD>    method to test for outliers [default: zscore] [possible values: zscore, dbscan]\n"
                   "  -s, --sample <SAMPLE>    sample to consider\n  -S, --subset <SUBSET>    file with subset of samples to consider\n"
                   "  -h, --help               Print help\n", usage);
            return 0;
        } else if (!a.empty() && a[0] == '-' && a.size() > 1) cusage("unexpected argument '" + a + "' found", usage);
        else if (combined.empty()) combined = a;
        else cusage("unexpected argument '" + a + "' found", usage);
    }
    if (combined.empty()) cusage("the following required arguments were not provided:\n  <COMBINED>", usage);
    if (!exists(combined)) cpanic("Combined file does not exist!");                       // main.rs:210-212
    if (has_sample && has_subset) cpanic("Cannot use both -s and -S arguments");          // main.rs:214-216
    std::unordered_set<std::string> subset;
    const bool use_subset = has_sample || has_subset;
    if (has_sample) subset.insert(sample);
    if (has_subset) {
        LineReader sr;
        if (!sr.open(subset_file)) cpanic("Problem opening file");                        // utils.rs:9
        std::string l;
        while (sr.next(l)) subset.insert(l);
    }

    LineReader rd;
    if (!rd.open(combined)) cpanic("Problem opening file");
    std::string line;
    if (!rd.next(line)) cpanic("called `Option::unwrap()` on a `None` value");            // outlier.rs:36
    fputs("chrom\tbegin\tend\toutliers\n", stdout);                                       // outlier.rs:37
    std::vector<std::string> cols;
    split_tabs(line, cols);
    std::vector<std::string> samples(cols.begin() + std::min<size_t>(3, cols.size()), cols.end());
    if (samples.empty()) cpanic("argument of integer logarithm must be positive");       // ilog2(0), outlier.rs:39
    const uint32_t n_cols = (uint32_t)samples.size();
    std::vector<std::string> names(n_cols);
    for (uint32_t c = 0; c < n_cols; ++c) names[c] = strip_hap(samples[c]);
    const int meth = method == "dbscan" ? INQ_OUTLIER_DBSCAN : INQ_OUTLIER_ZSCORE;

    // rows are processed in batches of the combined matrix
    const size_t batch_rows = std::max<size_t>(1, std::min<size_t>(1u << 16, (256u << 20) / ((size_t)n_cols * sizeof(float))));
    std::vector<float> values;
    std::vector<std::string> keys;                       // "chrom\tbegin\tend"
    std::vector<uint64_t> hits;
    auto flush = [&]() {
        uint64_t rows = keys.size();
        if (!rows) return;
        uint64_t n_hits = 0;
        if (hits.size() < 1024) hits.resize(1024);
        int rc;
        std::string no_mode;
        for (;;) {
            while ((rc = inq_outlier(device, meth, rows, n_cols, values.data(), (uint32_t)minsize, zscore, nullptr, &n_hits,
                                     hits.data(), hits.size(), nullptr)) == INQ_ERR_HITS_CAP)
                hits.resize(n_hits);
            if (rc != INQ_ERR_NO_MODE || !no_mode.empty()) break;
            // The reference streams row by row: the rows before the one without a mode have been printed when it panics
            // (outlier.rs:144). The message names a row without a mode; the batch is cut at the FIRST one.
            no_mode = inq_cohort_last_error();
            const size_t at = no_mode.find("row ");
            uint64_t bad = at == std::string::npos ? 0 : strtoull(no_mode.c_str() + at + 4, nullptr, 10);
            // rows are independent: find the first bad row by re-running ever shorter prefixes (rare path)
            while (bad > 0) {
                uint64_t nh = 0;
                const int r2 = inq_outlier(device, meth, bad, n_cols, values.data(), (uint32_t)minsize, zscore, nullptr, &nh, hits.data(), 0, nullptr);
                if (r2 != INQ_ERR_NO_MODE) break;
                const std::string m2 = inq_cohort_last_error();
                const size_t a2 = m2.find("row ");
                const uint64_t b2 = a2 == std::string::npos ? 0 : strtoull(m2.c_str() + a2 + 4, nullptr, 10);
                if (b2 >= bad) break;
                bad = b2;
            }
            rows = bad;
            if (!rows) break;
        }
        if (rc == INQ_ERR_NO_MODE) cpanic(std::string("No mode found for repeat (") + no_mode + ")");          // the first row of the batch
        if (rc != INQ_OK) { fprintf(stderr, "inquistr-b200: %s\n", inq_cohort_last_error()); exit(1); }
        if (rc != INQ_OK) { fprintf(stderr, "inquistr-b200: %s\n", inq_cohort_last_error()); exit(1); }
        std::string out;
        for (uint64_t i = 0; i < n_hits;) {
            const uint64_t row = hits[i] >> 32;
            uint64_t j = i;
            bool wanted = !use_subset;
            out = keys[row];
            out.push_back('\t');
            for (; j < n_hits && (hits[j] >> 32) == row; ++j) {
                const std::string &nm = names[hits[j] & 0xFFFFFFFFull];
                if (j > i) out.push_back(',');
                out += nm;
                if (use_subset && subset.count(nm)) wanted = true;                        // outlier.rs:59-64
            }
            out.push_back('\n');
            if (wanted) fwrite(out.data(), 1, out.size(), stdout);
            i = j;
        }
        if (!no_mode.empty()) { fflush(stdout); cpanic(std::string("No mode found for repeat (") + no_mode + ")"); }   // outlier.rs:144
        values.clear();
        keys.clear();
    };
    while (rd.next(line)) {
        split_tabs(line, cols);
        // the reference prints row by row, so everything before a row it panics on is already out: flush first
        auto die = [&](const std::string &msg) { values.resize(keys.size() * (size_t)n_cols); flush(); fflush(stdout); cpanic(msg); };
        if (cols.size() < 3) die("index out of bounds: the len is " + std::to_string(cols.size()) + " but the index is 2");
        if (cols.size() - 3 > n_cols) die("index out of bounds: more values than samples in the header");
        if (cols.size() - 3 < n_cols)
            die("row '" + cols[0] + "\t" + cols[1] + "\t" + cols[2] + "' has fewer values than the header has samples (this build needs a rectangular matrix)");
        for (uint32_t c = 0; c < n_cols; ++c) {
            float f;
            if (!parse_f32(cols[3 + c], &f)) die("Failed to parse number: ParseFloatError { kind: Invalid }");   // outlier.rs:79
            values.push_back(f);
        }
        keys.push_back(cols[0] + "\t" + cols[1] + "\t" + cols[2]);
        if (keys.size() == batch_rows) flush();
    }
    flush();
    return 0;
}

namespace {

[[noreturn]] void afail(const std::string &msg)
{
    fflush(stdout);
    fprintf(stderr, "inquistr-b200: %s\n", msg.c_str());
    exit(1);
}

// a finite decimal number, the whole field
bool parse_f64(const std::string &s, double *out)
{
    if (s.empty() || isspace((unsigned char)s[0])) return false;
    char *end = nullptr;
    *out = strtod(s.c_str(), &end);
    return end && *end == '\0' && std::isfinite(*out);
}

// a value of the combined table: a finite number or NaN (no call)
bool parse_call(const std::string &s, double *out)
{
    if (s.size() == 3 && tolower((unsigned char)s[0]) == 'n' && tolower((unsigned char)s[1]) == 'a' && tolower((unsigned char)s[2]) == 'n') {
        *out = NAN;
        return true;
    }
    return parse_f64(s, out);
}

void append_f64(std::string &out, double v)
{
    if (std::isnan(v)) { out += "NaN"; return; }
    char buf[64];
    const auto r = std::to_chars(buf, buf + sizeof(buf), v);          // shortest form that round-trips
    out.append(buf, r.ptr);
}

}  // namespace

// `assoc`: one regression per row of a combined table (DESIGN.md 5e)
int assoc_main(const std::vector<std::string> &v, int device)
{
    const char *usage = "assoc --phenotype <TSV> --trait <COL> | --traits <A,B,...> --model <linear|logistic|cox> [--firth] [--event <COL>] [--ties efron|breslow] [--covariates A,B,...] [--predictor sum|max] [--device N] <COMBINED>";
    std::string combined, pheno, trait, model, predictor = "sum", covs, trait_list, stats_json, event_col, ties;
    bool has_cov = false, firth = false, has_traits = false, has_event = false;
    for (size_t i = 0; i < v.size(); ++i) {
        const std::string &a = v[i];
        auto value = [&](const char *name) -> std::string {
            if (i + 1 >= v.size()) cusage(std::string("a value is required for '") + name + "' but none was supplied", usage);
            return v[++i];
        };
        if (a == "--phenotype") pheno = value("--phenotype <TSV>");
        else if (a == "--trait") trait = value("--trait <COL>");
        else if (a == "--traits") { trait_list = value("--traits <A,B,...>"); has_traits = true; }
        else if (a == "--model") {
            model = value("--model <MODEL>");
            if (model != "linear" && model != "logistic" && model != "cox") cusage("invalid value '" + model + "' for '--model <MODEL>'\n  [possible values: linear, logistic, cox]", usage);
        } else if (a == "--firth") firth = true;
        else if (a == "--event") { event_col = value("--event <COL>"); has_event = true; }
        else if (a == "--ties") {
            ties = value("--ties <TIES>");
            if (ties != "efron" && ties != "breslow") cusage("invalid value '" + ties + "' for '--ties <TIES>'\n  [possible values: efron, breslow]", usage);
        }
        else if (a == "--covariates") { covs = value("--covariates <A,B,...>"); has_cov = true; }
        else if (a == "--predictor") {
            predictor = value("--predictor <PREDICTOR>");
            if (predictor != "sum" && predictor != "max") cusage("invalid value '" + predictor + "' for '--predictor <PREDICTOR>'\n  [possible values: sum, max]", usage);
        } else if (a == "--device") {
            const std::string s = value("--device <N>");
            char *e = nullptr;
            const long d = strtol(s.c_str(), &e, 10);
            if (s.empty() || *e || d < 0 || d > 1024) cusage("invalid value '" + s + "' for '--device <N>'", usage);
            device = (int)d;
        } else if (a == "--stats-json") stats_json = value("--stats-json <FILE>");
        else if (a == "-h" || a == "--help") {
            printf("Test every locus of a combined table for association with a phenotype\n\nUsage: inquistr-b200 %s\n\n"
                   "Arguments:\n  <COMBINED>  combined table of calls (`call-cohort` or `combine` output, plain or gzip)\n\nOptions:\n"
                   "      --phenotype <TSV>        tab-separated phenotype table with a header; first column: sample names\n"
                   "      --trait <COL>            response column\n"
                   "      --traits <A,B,...>       several response columns in one run (instead of --trait); a sample with a missing\n"
                   "                               value (NA, NaN, empty) is left out for that trait only\n"
                   "      --model <MODEL>          linear (OLS, t test) or logistic (0/1 trait, IRLS, Wald z test) [possible values: linear, logistic]\n"
                   "                               or cox (Cox proportional hazards, Wald z test): --trait is the time (age at onset or at\n"
                   "                               last visit), --event the event column\n"
                   "      --event <COL>            with --model cox: 1 = event (onset) at the time, 0 = censored (no onset yet)\n"
                   "      --ties <TIES>            with --model cox: tied event times [default: efron] [possible values: efron, breslow]\n"
                   "      --firth                  with --model logistic: Firth-penalized fit (finite under separation) and\n"
                   "                               penalized likelihood-ratio test\n"
                   "      --covariates <A,B,...>   0 to %d covariate columns; samples with a missing value (NA, NaN, empty) are left out\n"
                   "      --predictor <PREDICTOR>  per sample and locus: H1 + H2, or the larger allele [default: sum] [possible values: sum, max]\n"
                   "      --device <N>             CUDA device [default: 0]\n"
                   "      --stats-json <FILE>      write parse, device and output times to FILE\n"
                   "  -h, --help                   Print help\n\n"
                   "Output: chromosome begin end n beta se stat p status, one row per input row; status is one of ok,\n"
                   "few_samples, singular, no_convergence, separation. With --traits: chromosome begin end trait n beta se stat\n"
                   "p status, one row per input row and trait in --traits order. With --firth, stat is the penalized likelihood-ratio\n"
                   "chi-square (1 df) of x, p comes from it, and separation is never reported. With --model cox, stat is the Wald z\n"
                   "of x and a sample missing its time or event is left out\n", usage, INQ_ASSOC_MAX_COV);
            return 0;
        } else if (!a.empty() && a[0] == '-' && a.size() > 1) cusage("unexpected argument '" + a + "' found", usage);
        else if (combined.empty()) combined = a;
        else cusage("unexpected argument '" + a + "' found", usage);
    }
    std::string missing;
    if (pheno.empty()) missing += "\n  --phenotype <TSV>";
    if (has_traits && !trait.empty()) cusage("the argument '--traits <A,B,...>' cannot be used with '--trait <COL>'", usage);
    if (trait.empty() && !has_traits) missing += "\n  --trait <COL>";
    if (model.empty()) missing += "\n  --model <MODEL>";
    if (combined.empty()) missing += "\n  <COMBINED>";
    if (!missing.empty()) cusage("the following required arguments were not provided:" + missing, usage);
    if (firth && model != "logistic") cusage("the argument '--firth' requires '--model logistic'", usage);
    const bool cox = model == "cox";
    if (has_event && !cox) cusage("the argument '--event <COL>' requires '--model cox'", usage);
    if (!ties.empty() && !cox) cusage("the argument '--ties <TIES>' requires '--model cox'", usage);
    if (cox && has_traits) cusage("the argument '--traits <A,B,...>' cannot be used with '--model cox'", usage);
    if (cox && !has_event) cusage("the following required arguments were not provided:\n  --event <COL> (with --model cox)", usage);
    if (cox && event_col == trait) cusage("the event column '" + event_col + "' is also the time column (--trait)", usage);
    auto split_list = [](const std::string &s) {
        std::vector<std::string> out;
        size_t a = 0;
        for (;;) {
            const size_t b = s.find(',', a);
            out.emplace_back(s, a, b == std::string::npos ? std::string::npos : b - a);
            if (b == std::string::npos) break;
            a = b + 1;
        }
        return out;
    };
    std::vector<std::string> cov_names, traits{trait};
    if (has_cov && !covs.empty()) cov_names = split_list(covs);
    if (has_traits) {
        traits = split_list(trait_list);
        for (size_t t = 0; t < traits.size(); ++t) {
            if (traits[t].empty()) cusage("invalid value '" + trait_list + "' for '--traits <A,B,...>': an empty column name", usage);
            for (size_t d = 0; d < t; ++d)
                if (traits[d] == traits[t]) cusage("trait '" + traits[t] + "' is listed twice", usage);
        }
    }
    if (cov_names.size() > INQ_ASSOC_MAX_COV)
        cusage("invalid value '" + covs + "' for '--covariates <A,B,...>': " + std::to_string(cov_names.size()) + " covariates, at most " +
               std::to_string(INQ_ASSOC_MAX_COV), usage);
    for (size_t c = 0; c < cov_names.size(); ++c) {
        if (cov_names[c].empty()) cusage("invalid value '" + covs + "' for '--covariates <A,B,...>': an empty column name", usage);
        for (const std::string &t : traits)
            if (cov_names[c] == t) cusage("the trait '" + t + "' is also listed as a covariate", usage);
        if (cox && cov_names[c] == event_col) cusage("the event column '" + event_col + "' is also listed as a covariate", usage);
        for (size_t d = 0; d < c; ++d)
            if (cov_names[d] == cov_names[c]) cusage("covariate '" + cov_names[c] + "' is listed twice", usage);
    }
    const bool logistic = model == "logistic";
    const auto t_start = std::chrono::steady_clock::now();

    // phenotype table: sample -> traits, covariates; rows with a missing covariate (or, for cox, event) are left out, a
    // missing trait value (NaN) leaves the sample out for that trait only
    const size_t n_cov = cov_names.size(), n_tr = traits.size(), n_ev = cox ? 1 : 0;
    std::unordered_map<std::string, std::vector<double>> ph;          // rows with every covariate: [traits..., event, covariates...]
    std::unordered_set<std::string> ph_seen;
    size_t cov_missing = 0;
    std::vector<size_t> ph_missing(n_tr, 0);                          // per trait: rows left out for it
    {
        LineReader pr;
        if (!exists(pheno) || !pr.open(pheno)) afail(pheno + ": cannot open the phenotype table");
        std::string line;
        std::vector<std::string> cols;
        if (!pr.next(line)) afail(pheno + ":1: empty file (a header row is needed)");
        split_tabs(line, cols);
        const std::vector<std::string> head = cols;
        std::vector<std::string> want_names = traits;                 // [traits..., event (cox), covariates...]
        if (cox) want_names.push_back(event_col);
        want_names.insert(want_names.end(), cov_names.begin(), cov_names.end());
        std::vector<size_t> want;
        for (const std::string &name : want_names) {
            size_t k = 1;
            while (k < head.size() && head[k] != name) ++k;
            if (k >= head.size()) afail(pheno + ":1: column '" + name + "' is not in the header");
            want.push_back(k);
        }
        for (uint64_t ln = 2; pr.next(line); ++ln) {
            if (line.empty()) continue;
            split_tabs(line, cols);
            const std::string where = pheno + ":" + std::to_string(ln) + ": ";
            if (cols.size() != head.size())
                afail(where + std::to_string(cols.size()) + " fields, the header has " + std::to_string(head.size()));
            if (!ph_seen.insert(cols[0]).second) afail(where + "column '" + head[0] + "': sample '" + cols[0] + "' appears twice");
            std::vector<double> vals(want.size(), NAN);
            bool complete = true;
            for (size_t w = 0; w < want.size(); ++w) {
                const std::string &f = cols[want[w]];
                if (f.empty() || f == "NA" || f == "NaN") { if (w >= n_tr) complete = false; continue; }
                if (!parse_f64(f, &vals[w])) afail(where + "column '" + head[want[w]] + "': '" + f + "' is not a number");
                if (w < n_tr && logistic && vals[w] != 0.0 && vals[w] != 1.0)
                    afail(where + "column '" + head[want[w]] + "': '" + f + "' is not 0 or 1 (--model logistic)");
                if (cox && w == n_tr && vals[w] != 0.0 && vals[w] != 1.0)
                    afail(where + "column '" + head[want[w]] + "': '" + f + "' is not 0 or 1 (--event)");
            }
            if (!complete) { ++cov_missing; continue; }
            bool any = false;
            for (size_t t = 0; t < n_tr; ++t) {
                if (std::isnan(vals[t])) ++ph_missing[t];
                else any = true;
            }
            if (any) ph.emplace(cols[0], std::move(vals));
        }
    }

    // combined table header: chromosome begin end <S>_H1 <S>_H2 ...
    if (!exists(combined)) afail(combined + ": no such file");
    LineReader rd;
    if (!rd.open(combined)) afail(combined + ": cannot open");
    std::string line;
    std::vector<std::string> cols;
    if (!rd.next(line)) afail(combined + ":1: empty file (a header row is needed)");
    split_tabs(line, cols);
    if (cols.size() < 3 || cols[0] != "chromosome" || cols[1] != "begin" || cols[2] != "end")
        afail(combined + ":1: the header does not start with 'chromosome begin end'");
    const size_t n_val = cols.size() - 3;
    if (n_val % 2) afail(combined + ":1: " + std::to_string(n_val) + " value columns: not in <S>_H1 <S>_H2 pairs");
    const size_t n_tab = n_val / 2;
    std::vector<uint32_t> use_idx;                       // table sample index of every sample used for some trait, in table order
    std::vector<double> y, cov;                          // y: use_idx.size() x n_tr, NaN = not used for that trait
    std::vector<uint8_t> event;                          // cox: the event of every sample used
    size_t n_groups = 0;
    {
        std::unordered_set<std::string> names;
        for (size_t k = 0; k < n_tab; ++k) {
            const std::string &h1 = cols[3 + 2 * k], &h2 = cols[4 + 2 * k];
            const bool pair = h1.size() > 3 && h2.size() == h1.size() && h1.compare(h1.size() - 3, 3, "_H1") == 0 &&
                              h2.compare(h2.size() - 3, 3, "_H2") == 0 && h1.compare(0, h1.size() - 3, h2, 0, h2.size() - 3) == 0;
            if (!pair) afail(combined + ":1: columns " + std::to_string(4 + 2 * k) + "-" + std::to_string(5 + 2 * k) + " ('" + h1 + "', '" + h2 +
                             "') are not a <S>_H1 <S>_H2 pair");
            const std::string s = h1.substr(0, h1.size() - 3);
            if (!names.insert(s).second) afail(combined + ":1: sample '" + s + "' appears twice");
            const auto it = ph.find(s);
            if (it == ph.end()) continue;
            use_idx.push_back((uint32_t)k);
            y.insert(y.end(), it->second.begin(), it->second.begin() + n_tr);
            if (cox) event.push_back((uint8_t)it->second[n_tr]);
            cov.insert(cov.end(), it->second.begin() + n_tr + n_ev, it->second.end());
        }
        size_t ph_only = 0;
        for (const std::string &s : ph_seen) ph_only += !names.count(s);
        std::vector<size_t> used(n_tr, 0);
        std::vector<std::vector<bool>> masks;            // the traits' sample sets, as inq_assoc_traits groups them
        for (size_t t = 0; t < n_tr; ++t) {
            std::vector<bool> m(use_idx.size());
            for (size_t s = 0; s < use_idx.size(); ++s) used[t] += m[s] = !std::isnan(y[s * n_tr + t]);
            if (std::find(masks.begin(), masks.end(), m) == masks.end()) masks.push_back(std::move(m));
        }
        n_groups = masks.size();
        if (!has_traits) {
            fprintf(stderr, "assoc: %zu samples used, %zu in the table only, %zu in the phenotype table only (%zu phenotype rows with a missing value left out)\n",
                    use_idx.size(), n_tab - use_idx.size(), ph_only, cov_missing + ph_missing[0]);
            if (use_idx.empty()) afail("no sample is in both " + combined + " and " + pheno);
        } else {
            for (size_t t = 0; t < n_tr; ++t)
                fprintf(stderr, "assoc: trait '%s': %zu samples used, %zu in the table only, %zu in the phenotype table only (%zu phenotype rows with a missing value left out)\n",
                        traits[t].c_str(), used[t], n_tab - used[t], ph_only, cov_missing + ph_missing[t]);
            for (size_t t = 0; t < n_tr; ++t)
                if (!used[t]) afail("trait '" + traits[t] + "': no sample is in both " + combined + " and " + pheno);
        }
    }
    const uint32_t ns = (uint32_t)use_idx.size();
    fputs(has_traits ? "chromosome\tbegin\tend\ttrait\tn\tbeta\tse\tstat\tp\tstatus\n" : "chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus\n", stdout);
    const char *status_names[] = {"ok", "few_samples", "singular", "no_convergence", "separation"};
    const int mdl = firth ? INQ_ASSOC_FIRTH : logistic ? INQ_ASSOC_LOGISTIC : INQ_ASSOC_LINEAR, prd = predictor == "max" ? INQ_ASSOC_MAX : INQ_ASSOC_SUM;
    const int tie = ties == "breslow" ? INQ_COX_BRESLOW : INQ_COX_EFRON;

    // rows in batches of at most 256 MB of values and 64 MB of results (rows x traits x 38 bytes)
    const size_t batch_rows = std::max<size_t>(1, std::min((256u << 20) / ((size_t)ns * 2 * sizeof(double)), (64u << 20) / (n_tr * 38)));
    std::vector<double> haps, beta, se, stat, pv, rowvals(n_val);
    std::vector<uint32_t> n_used;
    std::vector<uint8_t> status;
    std::vector<std::string> keys;
    double s_device = 0.0, s_write = 0.0;
    uint64_t n_rows = 0;
    std::string out;
    auto flush = [&]() {
        const size_t rows = keys.size();
        if (!rows) return;
        const size_t cells = rows * n_tr;
        beta.resize(cells); se.resize(cells); stat.resize(cells); pv.resize(cells); n_used.resize(cells); status.resize(cells);
        const auto t0 = std::chrono::steady_clock::now();
        const int rc = cox
            ? inq_assoc_cox(device, tie, prd, rows, ns, haps.data(), y.data(), event.data(), (uint32_t)n_cov, n_cov ? cov.data() : nullptr,
                            beta.data(), se.data(), stat.data(), pv.data(), n_used.data(), status.data(), nullptr, nullptr)
            : has_traits
            ? inq_assoc_traits(device, mdl, prd, rows, ns, haps.data(), (uint32_t)n_tr, y.data(), (uint32_t)n_cov, n_cov ? cov.data() : nullptr,
                               beta.data(), se.data(), stat.data(), pv.data(), n_used.data(), status.data(), nullptr, nullptr)
            : inq_assoc(device, mdl, prd, rows, ns, haps.data(), y.data(), (uint32_t)n_cov, n_cov ? cov.data() : nullptr,
                        beta.data(), se.data(), stat.data(), pv.data(), n_used.data(), status.data(), nullptr, nullptr);
        const auto t1 = std::chrono::steady_clock::now();
        s_device += std::chrono::duration<double>(t1 - t0).count();
        if (rc != INQ_OK) afail(inq_cohort_last_error());
        out.clear();
        for (size_t c = 0; c < cells; ++c) {
            out += keys[c / n_tr];
            out.push_back('\t');
            if (has_traits) { out += traits[c % n_tr]; out.push_back('\t'); }
            out += std::to_string(n_used[c]);
            for (double x : {beta[c], se[c], stat[c], pv[c]}) { out.push_back('\t'); append_f64(out, x); }
            out.push_back('\t');
            out += status[c] < 5 ? status_names[status[c]] : "?";
            out.push_back('\n');
            if (out.size() >= (4u << 20)) { fwrite(out.data(), 1, out.size(), stdout); out.clear(); }
        }
        fwrite(out.data(), 1, out.size(), stdout);
        s_write += std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
        n_rows += rows;
        haps.clear();
        keys.clear();
    };
    for (uint64_t ln = 2; rd.next(line); ++ln) {
        split_tabs(line, cols);
        const std::string where = combined + ":" + std::to_string(ln) + ": ";
        if (cols.size() != 3 + n_val) {
            flush();
            afail(where + std::to_string(cols.size() < 3 ? 0 : cols.size() - 3) + " values, the header has " + std::to_string(n_val));
        }
        for (size_t c = 0; c < n_val; ++c)
            if (!parse_call(cols[3 + c], &rowvals[c])) {
                flush();
                afail(where + "column " + std::to_string(4 + c) + ": '" + cols[3 + c] + "' is not a number");
            }
        for (uint32_t k : use_idx) { haps.push_back(rowvals[2 * k]); haps.push_back(rowvals[2 * k + 1]); }
        keys.push_back(cols[0] + "\t" + cols[1] + "\t" + cols[2]);
        if (keys.size() == batch_rows) flush();
    }
    flush();
    fflush(stdout);
    if (!stats_json.empty()) {
        const double total = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
        FILE *f = fopen(stats_json.c_str(), "w");
        if (!f) afail(stats_json + ": cannot write");
        fprintf(f, "{\"rows\": %llu, \"samples_used\": %u, \"traits\": %zu, \"groups\": %zu, \"s_total\": %.6f, \"s_device\": %.6f, \"s_write\": %.6f, \"s_parse\": %.6f}\n",
                (unsigned long long)n_rows, ns, n_tr, n_groups, total, s_device, s_write, total - s_device - s_write);
        fclose(f);
    }
    return 0;
}

}  // namespace inqhost
