// cohort_call.cpp -- `inquistr-b200 call-cohort`: `call` on several BAMs against one locus catalog in one process.
// stdout is byte-identical to `combine <(call ... BAM1) ... <(call ... BAMn)` run with the same options, but
//   * the catalog is parsed, validated against every BAM header and sorted once;
//   * each listed device gets one context (ShardWorker) that holds the whole catalog and genotypes the samples it
//     takes one after the other (push, inq_genotype, inq_clear_reads); the context and the catalog upload are paid
//     once per device, not once per sample;
//   * a free device takes the next unstarted sample in list order; the next BAM is read while the previous sample
//     is genotyped; results are kept by sample index as integers and formatted once at the end.
// Nothing on the device differs from `call`: each sample is one pass of the same kernels over the same catalog.
// Every error exits like the shell pipeline would fail (1 for an unusable input or device, 101 for a panic of the
// reference), and stdout stays empty: the table is printed only once every sample is done.
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cinttypes>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <unordered_set>
#include <vector>

#include <sys/stat.h>

#include "../../../include/inqcall.h"
#include "bam_reader.hpp"
#include "call_common.hpp"
#include "shard_driver.hpp"

namespace inqhost {

namespace {

const char *kCohortUsage = "inquistr-b200 call-cohort [OPTIONS] <BAM> <BAM>...";
const char *kCohortHelp =
    "Call lengths in several bams against one catalog and print the combined table\n"
    "(the output of `combine` over one `call` per bam, with one CUDA context per device)\n\n"
    "Usage: inquistr-b200 call-cohort [OPTIONS] <BAM> <BAM>...\n\n"
    "Arguments:\n"
    "  <BAM>...  bam files to call STRs in; the sample names are their file stems\n\n"
    "Options:\n"
    "  -r, --region <REGION>            region string to genotype expansion in\n"
    "  -R, --region-file <REGION_FILE>  Bed file with region(s) to genotype expansion(s) in\n"
    "  -m, --minlen <MINLEN>            minimal length of insertion/deletion operation [default: 5]\n"
    "  -s, --support <SUPPORT>          minimal number of supporting reads [default: 3]\n"
    "  -t, --threads <THREADS>          Number of parallel threads to use [default: 1]\n"
    "  -u, --unphased                   If reads have to be considered unphased\n"
    "      --devices <A,B,...>          CUDA devices, one context each; samples are spread over them [default: 0]\n"
    "      --stats-json <FILE>          write per-sample counters and timings as JSON\n"
    "  -h, --help                       Print help\n\n"
    "The results of every sample are held in memory until all are done: 17 bytes per locus and sample\n"
    "(1M loci x 268 samples: 4.6 GB).\n";

[[noreturn]] void cohort_usage(const std::string &msg)
{
    fprintf(stderr, "error: %s\n\nUsage: %s\n\nFor more information, try '--help'.\n", msg.c_str(), kCohortUsage);
    exit(2);
}

struct CohortArgs {
    std::vector<std::string> bams;
    bool has_region = false, has_region_file = false;
    std::string region, region_file;
    uint32_t minlen = 5;
    uint64_t support = 3, threads = 1;
    bool unphased = false;
    std::vector<int> devices;
    std::string stats_json;
};

// the option syntax of `call` (main.cpp parse_args), without --sample-name / --reference / --device
CohortArgs parse_cohort_args(const std::vector<std::string> &v, std::vector<int> devices)
{
    if (v.empty()) { fputs(kCohortHelp, stderr); exit(2); }
    CohortArgs a;
    a.devices = std::move(devices);
    auto need = [&](size_t &i, const std::string &name) -> std::string {
        if (i + 1 >= v.size()) cohort_usage("a value is required for '" + name + "' but none was supplied");
        return v[++i];
    };
    auto set_opt = [&](const std::string &name, const std::string &val) {
        uint64_t n = 0;
        if (name == "region") { a.region = val; a.has_region = true; }
        else if (name == "region-file") { a.region_file = val; a.has_region_file = true; }
        else if (name == "minlen") { if (!parse_u64(val, &n) || n > UINT32_MAX) cohort_usage("invalid value '" + val + "' for '--minlen <MINLEN>'"); a.minlen = (uint32_t)n; }
        else if (name == "support") { if (!parse_u64(val, &n)) cohort_usage("invalid value '" + val + "' for '--support <SUPPORT>'"); a.support = n; }
        else if (name == "threads") { if (!parse_u64(val, &n)) cohort_usage("invalid value '" + val + "' for '--threads <THREADS>'"); a.threads = n; }
        else if (name == "devices") { if (!parse_device_list(val, &a.devices)) cohort_usage("invalid value '" + val + "' for '--devices <A,B,...>'"); }
        else if (name == "stats-json") a.stats_json = val;
        else cohort_usage("unexpected argument '--" + name + "' found");
    };
    const std::map<char, std::string> shorts = {{'r', "region"}, {'R', "region-file"}, {'m', "minlen"}, {'s', "support"}, {'t', "threads"}};
    bool only_positional = false;
    for (size_t i = 0; i < v.size(); ++i) {
        const std::string &s = v[i];
        if (!only_positional && s == "--") { only_positional = true; continue; }
        if (!only_positional && s.rfind("--", 0) == 0) {
            std::string name = s.substr(2), val;
            const size_t eq = name.find('=');
            if (name == "help") { fputs(kCohortHelp, stdout); exit(0); }
            if (name == "unphased") { a.unphased = true; continue; }
            if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); }
            else if (name == "region" || name == "region-file" || name == "minlen" || name == "support" || name == "threads" ||
                     name == "devices" || name == "stats-json") val = need(i, "--" + name);
            set_opt(name, val);
        } else if (!only_positional && s.size() >= 2 && s[0] == '-') {
            for (size_t k = 1; k < s.size(); ++k) {
                const char c = s[k];
                if (c == 'u') { a.unphased = true; continue; }
                if (c == 'h') { fputs(kCohortHelp, stdout); exit(0); }
                auto it = shorts.find(c);
                if (it == shorts.end()) cohort_usage(std::string("unexpected argument '-") + c + "' found");
                std::string val = s.substr(k + 1);
                if (!val.empty() && val[0] == '=') val = val.substr(1);
                if (val.empty()) val = need(i, std::string("-") + c);
                set_opt(it->second, val);
                break;
            }
        } else {
            a.bams.push_back(s);
        }
    }
    if (a.bams.empty()) cohort_usage("the following required arguments were not provided:\n  <BAM>...");
    return a;
}

// The catalog in the contig space of the names it uses: contig c of the catalog is the c-th of those names in the
// first BAM's header order, and each BAM maps its own tids onto it by name.
struct Catalog {
    std::vector<Locus> loci;                 // BED order; Locus::tid is the catalog contig
    std::vector<std::string> contigs;
    std::vector<uint32_t> order;             // catalog position -> BED index, sorted by (contig, start)
    std::vector<int64_t> contig_off;
    std::vector<int32_t> lstart, lend;
};

Catalog build_catalog(const CohortArgs &a, const std::vector<BamHeader> &hdrs)
{
    Catalog cat;
    // call.rs:182-202 against the first header, then repeats.rs:96-115's contig test against every other header
    if (a.has_region && !a.has_region_file) cat.loci.push_back(parse_region(a.region, hdrs[0]));
    else if (!a.has_region && a.has_region_file) cat.loci = parse_bed(a.region_file, hdrs[0]);
    else {
        fprintf(stderr, "ERROR: Specify a region string (-r) or a region_file (-R)!\n\n");
        exit(1);
    }
    for (size_t k = 1; k < hdrs.size(); ++k)
        for (const Locus &l : cat.loci) {
            const int tid = hdrs[k].tid(l.chrom);
            if (tid < 0 || (int64_t)l.end >= hdrs[k].ref_lens[tid]) panic_bad_contig(l.chrom);
        }
    for (const Locus &l : cat.loci)
        if (l.start < 10) panic("attempt to subtract with overflow (locus " + l.chrom + ":" + std::to_string(l.start) + " has start < 10, call.rs:285)");
    if (a.support > UINT32_MAX) panic("support does not fit the device counter");

    std::vector<int> cid_of_tid(hdrs[0].ref_names.size(), -1);
    for (const Locus &l : cat.loci) cid_of_tid[l.tid] = 0;
    for (size_t t = 0; t < cid_of_tid.size(); ++t)
        if (cid_of_tid[t] == 0) { cid_of_tid[t] = (int)cat.contigs.size(); cat.contigs.push_back(hdrs[0].ref_names[t]); }
    for (Locus &l : cat.loci) l.tid = cid_of_tid[l.tid];

    // sorted by (contig, start); ties keep BED order
    const size_t L = cat.loci.size();
    const int n_contigs = (int)cat.contigs.size();
    cat.order.resize(L);
    std::iota(cat.order.begin(), cat.order.end(), 0u);
    std::stable_sort(cat.order.begin(), cat.order.end(), [&](uint32_t x, uint32_t y) {
        if (cat.loci[x].tid != cat.loci[y].tid) return cat.loci[x].tid < cat.loci[y].tid;
        return cat.loci[x].start < cat.loci[y].start;
    });
    cat.contig_off.assign(n_contigs + 1, 0);
    cat.lstart.resize(L);
    cat.lend.resize(L);
    for (size_t i = 0; i < L; ++i) {
        const Locus &l = cat.loci[cat.order[i]];
        cat.contig_off[l.tid + 1]++;
        cat.lstart[i] = (int32_t)l.start;
        cat.lend[i] = (int32_t)l.end;
    }
    for (int c = 0; c < n_contigs; ++c) cat.contig_off[c + 1] += cat.contig_off[c];
    return cat;
}

// The first error of the run by sample index; once one is raised the readers stop and no new sample starts.
struct FirstError {
    std::mutex mu;
    bool set = false;
    size_t sample = 0;
    int code = 0;
    std::string text;
    std::atomic<bool> abort{false};
    void raise(size_t s, int exit_code, const std::string &msg)
    {
        std::lock_guard<std::mutex> g(mu);
        if (!set || s < sample) { set = true; sample = s; code = exit_code; text = msg; }
        abort = true;
    }
    void panic(size_t s, const std::string &msg) { raise(s, 101, "thread 'main' panicked: " + msg + "\n"); }
    void library(size_t s, int rc, const std::string &msg)        // as main.cpp reports a failed shard
    {
        if (rc == INQ_ERR_BAD_HP || rc == INQ_ERR_BAD_SA || rc == INQ_ERR_MEDIAN_EMPTY || rc == INQ_ERR_LOCUS_START) panic(s, msg);
        else raise(s, 1, "ERROR: " + msg + " (code " + std::to_string(rc) + ")\n");
    }
};

struct SampleStats {
    bool used_index = false;
    uint64_t records = 0, pushed = 0, unpairable = 0, bytes_inflated = 0;
    double s_scan = 0;
    int slot = -1;
};

// call's HP decoding (get_phase, call.rs:349,482-491; see consider() in main.cpp): false for the aux type the
// reference panics on
bool decode_hp(bool unphased, HpType type, int64_t value, uint8_t *hp)
{
    *hp = 0xFF;
    if (unphased) return true;
    switch (type) {
    case HpType::Absent: return true;
    case HpType::U8:
    case HpType::I32: *hp = (uint8_t)value; break;
    default: return false;
    }
    if (*hp == 0xFF) *hp = 0xFE;
    return true;
}

struct Cohort {
    const CohortArgs &args;
    const Catalog &cat;
    const std::vector<BamHeader> &hdrs;
    int host_threads;                       // per reader
    FirstError err;
    std::vector<SampleStats> stats;
    std::vector<ShardResult> results;

    // One sample into a worker: the records `call` would push, with tids mapped to the catalog's contigs.
    // false when an error was raised.
    bool scan(size_t s, ShardWorker &w)
    {
        const std::string &path = args.bams[s];
        const BamHeader &h = hdrs[s];
        SampleStats &st = stats[s];
        const int n_contigs = (int)cat.contigs.size();
        std::vector<int> cid(h.ref_names.size(), -1), tid(n_contigs, -1);
        for (int c = 0; c < n_contigs; ++c) { tid[c] = h.tid(cat.contigs[c]); cid[tid[c]] = c; }

        // the .bai rule of `call` (main.cpp): windows closer than 100 kb fetched as one region
        std::vector<std::array<int64_t, 3>> regions;
        int64_t region_span = 0, genome = 0;
        for (int64_t len : h.ref_lens) genome += len;
        for (int c = 0; c < n_contigs; ++c)
            for (int64_t i = cat.contig_off[c]; i < cat.contig_off[c + 1]; ++i) {
                const int64_t b = (int64_t)cat.lstart[i] - 10, e = (int64_t)cat.lend[i] + 10;
                if (!regions.empty() && regions.back()[0] == tid[c] && b <= regions.back()[2] + 100000) regions.back()[2] = std::max(regions.back()[2], e);
                else regions.push_back({(int64_t)tid[c], b, e});
            }
        for (const auto &r : regions) region_span += r[2] - r[1] + 50000;
        std::string bai = path + ".bai";
        if (!is_file(bai) && ends_with(path, ".bam")) bai = path.substr(0, path.size() - 4) + ".bai";
        const char *idx_env = getenv("INQ_BAM_INDEX");
        const bool want_index = idx_env ? atoi(idx_env) != 0 : (region_span * 10 < genome);
        st.used_index = want_index && is_file(bai);

        auto push = [&](int c, int32_t pos, int32_t end, uint8_t mapq, uint8_t hp, uint8_t fl, const uint32_t *cig, uint32_t n_cig) {
            if (mapq <= 10 || (!args.unphased && hp == 0xFF)) { ++st.unpairable; return; }
            w.add(c, pos, end, mapq, hp, fl, cig, n_cig);
            ++st.pushed;
        };

        if (st.used_index) {
            BamIndexedReader ibam;
            if (!ibam.open_bam(path)) { err.panic(s, "Error opening local BAM: " + ibam.error()); return false; }
            if (!ibam.load_index(bai)) { err.panic(s, "Error opening BAM index: " + ibam.error()); return false; }
            std::unordered_set<uint64_t> seen;
            bool bad_hp = false;
            for (const auto &r : regions) {
                if (bad_hp || err.abort || w.failed()) break;
                const bool ok = ibam.fetch((int)r[0], r[1], r[2], [&](const BamRecordView &rec, uint64_t voff) {
                    ++st.records;
                    if (bad_hp || !seen.insert(voff).second) return;
                    const int c = cid[rec.tid];
                    if (!w.reaches(c, rec.pos, rec.end)) return;
                    uint8_t hp;
                    if (!decode_hp(args.unphased, rec.hp_type, rec.hp_value, &hp)) { bad_hp = true; return; }
                    if (rec.mapq <= 10 || (!args.unphased && hp == 0xFF)) { ++st.unpairable; return; }
                    bool sa_panic = false, has_clip = false;
                    for (uint32_t i = 0; i < rec.n_cigar && !has_clip; ++i) has_clip = (rec.cigar[i] & 0xF) == 4;
                    const bool two_d = has_clip ? is_accidental_2d(rec, &sa_panic) : false;
                    push(c, rec.pos, rec.end, rec.mapq, hp, (uint8_t)((two_d ? INQ_FLAG_ACCIDENTAL_2D : 0) | (sa_panic ? INQ_FLAG_SA_PANIC : 0)),
                         rec.cigar, rec.n_cigar);
                });
                if (!ok) { err.panic(s, "Failed to fetch region: " + ibam.error()); return false; }
            }
            st.bytes_inflated = ibam.bytes_inflated();
            if (bad_hp) { err.panic(s, "Unexpected type of Aux for HP (call.rs:487)"); return false; }
            return !err.abort;
        }

        BamReader bam;
        const char *gi = getenv("INQ_GPU_INFLATE");
        struct stat bst;
        const bool big = stat(path.c_str(), &bst) == 0 && (uint64_t)bst.st_size >= (2ull << 30);
        if (!bam.open(path, host_threads, (gi ? atoi(gi) != 0 : big) ? w.device() : -1)) { err.panic(s, "Error opening local BAM: " + bam.error()); return false; }
        struct ReachCtx { const std::vector<int> *cid; const ShardWorker *w; };
        const ReachCtx rctx{&cid, &w};
        RecFilter filt;
        filt.ctx = &rctx;
        filt.reach = [](const void *p, int32_t t, int32_t pos, int32_t end) {
            const ReachCtx &r = *static_cast<const ReachCtx *>(p);
            return t >= 0 && t < (int32_t)r.cid->size() && r.w->reaches((*r.cid)[t], pos, end);
        };
        filt.need_hp = !args.unphased;
        // two stages as in `call`: this thread inflates and parses, a routing thread pushes the parsed chunks in file order
        std::mutex qmu;
        std::condition_variable qcv;
        std::deque<std::vector<ParsedChunk>> parsed;
        bool parse_done = false, bad_hp = false;
        std::atomic<bool> dead{false};
        std::thread router([&] {
            for (;;) {
                std::vector<ParsedChunk> chunks;
                {
                    std::unique_lock<std::mutex> lk(qmu);
                    qcv.wait(lk, [&] { return !parsed.empty() || parse_done; });
                    if (parsed.empty()) return;
                    chunks = std::move(parsed.front());
                    parsed.pop_front();
                }
                qcv.notify_all();
                for (const ParsedChunk &pc : chunks) {
                    st.records += pc.n_records;
                    for (const BamRecLite &r : pc.recs) {
                        if (dead) break;
                        uint8_t hp;
                        if (!decode_hp(args.unphased, r.hp_type, r.hp_value, &hp)) { bad_hp = true; dead = true; break; }
                        const uint8_t fl = (uint8_t)((r.two_d ? INQ_FLAG_ACCIDENTAL_2D : 0) | (r.sa_panic ? INQ_FLAG_SA_PANIC : 0));
                        push(cid[r.tid], r.pos, r.end, r.mapq, hp, fl, r.cigar, r.n_cigar);
                    }
                }
                if (w.failed() || err.abort) dead = true;
            }
        });
        const int parse_threads = std::max(2, host_threads / 2);
        for (;;) {
            std::vector<ParsedChunk> chunks;
            if (dead || !bam.next_parsed(filt, parse_threads, chunks)) break;
            std::unique_lock<std::mutex> lk(qmu);
            qcv.wait(lk, [&] { return parsed.size() < 2; });
            parsed.push_back(std::move(chunks));
            lk.unlock();
            qcv.notify_all();
        }
        { std::lock_guard<std::mutex> lk(qmu); parse_done = true; }
        qcv.notify_all();
        router.join();
        st.bytes_inflated = bam.bytes_inflated();
        if (bad_hp) { err.panic(s, "Unexpected type of Aux for HP (call.rs:487)"); return false; }
        if (!bam.error().empty()) { err.panic(s, "Error reading BAM file: " + bam.error()); return false; }
        return !err.abort;
    }

    bool collect(size_t s, ShardWorker &w)
    {
        if (w.take_result(results[s])) return true;
        err.library(s, results[s].rc, results[s].error);
        return false;
    }

    // one device: the next unstarted sample while there is one; sample k+1 is read while sample k is genotyped
    void device_loop(int slot, ShardWorker &w, std::atomic<size_t> &next)
    {
        std::deque<size_t> pending;
        for (;;) {
            if (err.abort) break;
            const size_t s = next.fetch_add(1);
            if (s >= args.bams.size()) break;
            stats[s].slot = slot;
            const auto t0 = std::chrono::steady_clock::now();
            const bool ok = scan(s, w);
            stats[s].s_scan = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (!ok) return;
            w.end_sample();
            pending.push_back(s);
            while (pending.size() > 1) {
                if (!collect(pending.front(), w)) return;
                pending.pop_front();
            }
        }
        for (; !pending.empty() && !err.abort; pending.pop_front())
            if (!collect(pending.front(), w)) return;
    }
};

std::string json_str(const std::string &s)
{
    std::string o = "\"";
    for (char c : s) {
        if (c == '"' || c == '\\') { o += '\\'; o += c; }
        else if ((unsigned char)c < 0x20) { char b[8]; snprintf(b, sizeof(b), "\\u%04x", c); o += b; }
        else o += c;
    }
    return o + "\"";
}

}  // namespace

int cohort_call_main(const std::vector<std::string> &argv, std::vector<int> devices)
{
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
    const CohortArgs args = parse_cohort_args(argv, std::move(devices));
    const size_t S = args.bams.size();

    // call.rs:87-90 for every BAM before anything is read
    for (const std::string &bam : args.bams) {
        if (!is_file(bam) && !starts_with(bam, "s3") && !starts_with(bam, "https://")) {
            fprintf(stderr, "ERROR: path to bam file %s is not valid!\n\n", bam.c_str());
            return 1;
        }
        if (!is_file(bam)) {
            fprintf(stderr, "ERROR: remote input (%s) is not supported by this build (no libcurl/htslib); use a local BAM\n", bam.c_str());
            return 1;
        }
        if (ends_with(bam, ".cram")) {
            fprintf(stderr, "ERROR: CRAM input (%s) is not supported by this build (no htslib CRAM codec); convert to BAM\n", bam.c_str());
            return 1;
        }
    }
    // every header, then the catalog against all of them (call.rs:242-243, repeats.rs:96-115)
    std::vector<BamHeader> hdrs(S);
    for (size_t s = 0; s < S; ++s) {
        BamIndexedReader ibam;
        if (!ibam.open_bam(args.bams[s])) panic("Error opening local BAM: " + ibam.error());
        hdrs[s] = ibam.header();
    }
    const Catalog cat = build_catalog(args, hdrs);
    const size_t L = cat.loci.size();

    // one context per device, at most one per sample; each holds the whole catalog
    const size_t n_workers = std::min(args.devices.size(), S);
    const int total_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    Cohort co{args, cat, hdrs, std::max(1, total_threads / (int)n_workers)};
    co.stats.resize(S);
    co.results.resize(S);
    std::vector<std::unique_ptr<ShardWorker>> workers;
    for (size_t g = 0; g < n_workers; ++g)
        workers.emplace_back(new ShardWorker(args.devices[g], 0, L, (int)cat.contigs.size(), cat.contig_off, cat.lstart.data(), cat.lend.data(),
                                             args.minlen, (uint32_t)args.support, args.unphased, n_workers <= 2 ? 4 : 2));
    std::atomic<size_t> next{0};
    std::vector<std::thread> loops;
    for (size_t g = 0; g < n_workers; ++g) loops.emplace_back([&, g] { co.device_loop((int)g, *workers[g], next); });
    for (auto &t : loops) t.join();
    for (auto &w : workers) w->stop();
    if (co.err.set) {
        fputs(co.err.text.c_str(), stderr);
        return co.err.code;
    }

    // output order of `call`: -t 1 BED order (call.rs:149-157); -t > 1 sorted by (human chrom, start) (call.rs:137-145)
    std::vector<uint32_t> pos_of(L);
    for (size_t i = 0; i < L; ++i) pos_of[cat.order[i]] = (uint32_t)i;
    std::vector<uint32_t> out_order(L);
    std::iota(out_order.begin(), out_order.end(), 0u);
    if (args.threads > 1)
        std::stable_sort(out_order.begin(), out_order.end(), [&](uint32_t x, uint32_t y) {
            const int c = human_compare(cat.loci[x].chrom, cat.loci[y].chrom);
            if (c != 0) return c < 0;
            return cat.loci[x].start < cat.loci[y].start;
        });
    std::string out = "chromosome\tbegin\tend";
    for (const std::string &bam : args.bams) {
        const std::string name = sample_from_path(bam);
        out += "\t" + name + "_H1\t" + name + "_H2";
    }
    out += '\n';
    for (uint32_t bi : out_order) {
        const Locus &l = cat.loci[bi];
        const uint32_t p = pos_of[bi];
        out += l.chrom;
        out += '\t';
        out += std::to_string(l.start);
        out += '\t';
        out += std::to_string(l.end);
        for (size_t s = 0; s < S; ++s) {
            const ShardResult &r = co.results[s];
            out += '\t';
            out += fmt_phase(r.t1[p], r.valid[p] & INQ_VALID_H1);
            out += '\t';
            out += fmt_phase(r.t2[p], r.valid[p] & INQ_VALID_H2);
        }
        out += '\n';
        if (out.size() >= (4u << 20)) { fwrite(out.data(), 1, out.size(), stdout); out.clear(); }
    }
    fwrite(out.data(), 1, out.size(), stdout);
    fflush(stdout);

    if (!args.stats_json.empty()) {
        FILE *f = fopen(args.stats_json.c_str(), "w");
        if (f) {
            double s_ctx = 0;
            for (const ShardResult &r : co.results) s_ctx = std::max(s_ctx, r.s_ctx);
            fprintf(f, "{\"n_samples\": %zu, \"n_contexts\": %zu, \"n_loci\": %zu, \"s_ctx_create_set_loci\": %.3f, \"s_total\": %.3f, \"samples\": [",
                    S, n_workers, L, s_ctx, since(t_begin));
            for (size_t s = 0; s < S; ++s) {
                const SampleStats &st = co.stats[s];
                const ShardResult &r = co.results[s];
                fprintf(f, "%s{\"bam\": %s, \"context\": %d, \"used_index\": %d, \"records\": %" PRIu64 ", \"records_pushed\": %" PRIu64
                           ", \"records_unpairable\": %" PRIu64 ", \"bytes_inflated\": %" PRIu64 ", \"n_pairs\": %" PRIu64 ", \"ms_total\": %.4f"
                           ", \"s_bam_scan\": %.3f, \"s_genotype\": %.3f}",
                        s ? ", " : "", json_str(args.bams[s]).c_str(), st.slot, st.used_index ? 1 : 0, st.records, st.pushed, st.unpairable,
                        st.bytes_inflated, r.stats.n_pairs, r.stats.ms_total, st.s_scan, r.s_genotype);
            }
            fprintf(f, "]}\n");
            fclose(f);
        }
    }
    return 0;
}

}  // namespace inqhost
