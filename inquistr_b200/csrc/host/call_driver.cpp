// call_driver.cpp -- `inquistr-b200 call` and `inquistr-b200 call-cohort`: one host driver for both (the reference
// host is Rust; no Rust toolchain exists in this image, see INTEGRATION.md). Mirrors, above the C ABI of libinqcall.so:
//   CLI flags + defaults            src/main.rs:28-64
//   driver, sample name, header     src/call.rs:76-159
//   targets / validation            src/call.rs:161-202, src/repeats.rs:13-45,96-115
//   per-record fields               src/call.rs:297-299,349-352,415-459,482-491
//   ordering + row format           src/call.rs:27-65
// `call` is a run with one sample whose sorted catalog is cut over the listed devices (one ShardWorker context each,
// SURVEY 8e); `call-cohort` is a run with several samples over contexts that each hold the whole catalog. Both check
// every input, read every header, build one catalog, scan each sample and route every record to every worker that
// reaches it, collect the results and print one table. `call-cohort` prints the bytes of
// `combine <(call ... BAM1) ... <(call ... BAMn)` with the same options, but
//   * the catalog is parsed, validated against every BAM header and sorted once;
//   * each context genotypes the samples it takes one after the other (push, inq_genotype, inq_clear_reads), so the
//     context and the catalog upload are paid once per device, not once per sample;
//   * a free device takes the next unstarted sample in list order; the next BAM is read while the previous sample is
//     genotyped; results are kept by sample index as integers and formatted once at the end.
// stdout carries only the TSV, printed once every sample is done; diagnostics go to stderr. A Rust panic in the
// reference maps to exit code 101 here, `std::process::exit(1)` to 1, clap usage errors to 2; `call-cohort` exits
// as the shell pipeline would fail.
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

const char *kCallUsage = "inquistr-b200 call [OPTIONS] <BAM>";
const char *kCallHelp =
    "Call lengths\n\n"
    "Usage: inquistr-b200 call [OPTIONS] <BAM>\n\n"
    "Arguments:\n"
    "  <BAM>  bam file to call STRs in\n\n"
    "Options:\n"
    "  -r, --region <REGION>            region string to genotype expansion in\n"
    "  -R, --region-file <REGION_FILE>  Bed file with region(s) to genotype expansion(s) in\n"
    "  -m, --minlen <MINLEN>            minimal length of insertion/deletion operation [default: 5]\n"
    "  -s, --support <SUPPORT>          minimal number of supporting reads [default: 3]\n"
    "  -t, --threads <THREADS>          Number of parallel threads to use [default: 1]\n"
    "  -u, --unphased                   If reads have to be considered unphased\n"
    "      --sample-name <SAMPLE_NAME>  sample name to use in output\n"
    "      --reference <REFERENCE>      reference fasta for cram decoding\n"
    "      --device <N>                 (extension) CUDA device to run on [default: 0]\n"
    "      --devices <A,B,...>          (extension) shard the locus catalog over these CUDA devices (a device may repeat)\n"
    "      --stats-json <FILE>          (extension) write counters and device timings as JSON\n"
    "  -h, --help                       Print help\n";

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

struct CallArgs {
    bool cohort = false;
    std::vector<std::string> bams;
    bool has_region = false, has_region_file = false, has_sample = false;
    std::string region, region_file, sample_name;
    uint32_t minlen = 5;
    uint64_t support = 3, threads = 1;
    bool unphased = false;
    std::vector<int> devices;      // extension: CUDA devices (also INQ_DEVICE / INQ_DEVICES)
    std::string stats_json;        // extension: counters and timings side file
};

// clap's syntax for both subcommands. --sample-name, --reference and --device are `call`'s only; `call` takes exactly
// one BAM, `call-cohort` one or more.
CallArgs parse_call_args(const std::vector<std::string> &v, bool cohort, std::vector<int> devices)
{
    const char *usage = cohort ? kCohortUsage : kCallUsage;
    const char *help = cohort ? kCohortHelp : kCallHelp;
    if (v.empty()) { fputs(help, stderr); exit(2); }                     // arg_required_else_help (main.rs:27)
    CallArgs a;
    a.cohort = cohort;
    a.devices = std::move(devices);
    auto need = [&](size_t &i, const std::string &name) -> std::string {
        if (i + 1 >= v.size()) usage_error(usage, "a value is required for '" + name + "' but none was supplied");
        return v[++i];
    };
    auto takes_value = [&](const std::string &name) {
        return name == "region" || name == "region-file" || name == "minlen" || name == "support" || name == "threads" ||
               name == "devices" || name == "stats-json" || (!cohort && (name == "sample-name" || name == "reference" || name == "device"));
    };
    auto set_opt = [&](const std::string &name, const std::string &val) {
        uint64_t n = 0;
        if (!takes_value(name)) usage_error(usage, "unexpected argument '--" + name + "' found");
        if (name == "region") { a.region = val; a.has_region = true; }
        else if (name == "region-file") { a.region_file = val; a.has_region_file = true; }
        else if (name == "minlen") { if (!parse_u64(val, &n) || n > UINT32_MAX) usage_error(usage, "invalid value '" + val + "' for '--minlen <MINLEN>'"); a.minlen = (uint32_t)n; }
        else if (name == "support") { if (!parse_u64(val, &n)) usage_error(usage, "invalid value '" + val + "' for '--support <SUPPORT>'"); a.support = n; }
        else if (name == "threads") { if (!parse_u64(val, &n)) usage_error(usage, "invalid value '" + val + "' for '--threads <THREADS>'"); a.threads = n; }
        else if (name == "sample-name") { a.sample_name = val; a.has_sample = true; }
        else if (name == "device") { if (!parse_u64(val, &n)) usage_error(usage, "invalid value for '--device'"); a.devices.assign(1, (int)n); }
        else if (name == "devices") { if (!parse_device_list(val, &a.devices)) usage_error(usage, "invalid value '" + val + "' for '--devices <A,B,...>'"); }
        else if (name == "stats-json") a.stats_json = val;
        // --reference: accepted and unused, CRAM input is refused
    };
    const std::map<char, std::string> shorts = {{'r', "region"}, {'R', "region-file"}, {'m', "minlen"}, {'s', "support"}, {'t', "threads"}};
    bool only_positional = false;
    for (size_t i = 0; i < v.size(); ++i) {
        const std::string &s = v[i];
        if (!only_positional && s == "--") { only_positional = true; continue; }
        if (!only_positional && s.rfind("--", 0) == 0) {
            std::string name = s.substr(2), val;
            const size_t eq = name.find('=');
            if (name == "help") { fputs(help, stdout); exit(0); }
            if (name == "unphased") { a.unphased = true; continue; }
            if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); }
            else if (takes_value(name)) val = need(i, "--" + name);
            set_opt(name, val);
        } else if (!only_positional && s.size() >= 2 && s[0] == '-') {
            for (size_t k = 1; k < s.size(); ++k) {
                const char c = s[k];
                if (c == 'u') { a.unphased = true; continue; }
                if (c == 'h') { fputs(help, stdout); exit(0); }
                auto it = shorts.find(c);
                if (it == shorts.end()) usage_error(usage, std::string("unexpected argument '-") + c + "' found");
                std::string val = s.substr(k + 1);
                if (!val.empty() && val[0] == '=') val = val.substr(1);
                if (val.empty()) val = need(i, std::string("-") + c);
                set_opt(it->second, val);
                break;
            }
        } else {
            if (!cohort && !a.bams.empty()) usage_error(usage, "unexpected argument '" + s + "' found");
            a.bams.push_back(s);
        }
    }
    if (a.bams.empty()) usage_error(usage, std::string("the following required arguments were not provided:\n  ") + (cohort ? "<BAM>..." : "<BAM>"));
    return a;
}

// call.rs:87-90
void check_input(const std::string &bam)
{
    if (!is_file(bam) && !starts_with(bam, "s3") && !starts_with(bam, "https://")) {
        fprintf(stderr, "ERROR: path to bam file %s is not valid!\n\n", bam.c_str());
        exit(1);
    }
    if (!is_file(bam)) {
        fprintf(stderr, "ERROR: remote input (%s) is not supported by this build (no libcurl/htslib); use a local BAM\n", bam.c_str());
        exit(1);
    }
    if (ends_with(bam, ".cram")) {
        fprintf(stderr, "ERROR: CRAM input is not supported by this build (no htslib CRAM codec); convert %s to BAM\n", bam.c_str());
        exit(1);
    }
}

// The catalog in the contig space of the names it uses: contig c of the catalog is the c-th of those names in the
// first BAM's header order (so a coordinate-sorted BAM reaches the device sorted), and each BAM maps its own tids onto
// it by name.
struct Catalog {
    std::vector<Locus> loci;                 // BED order; Locus::tid is the catalog contig
    std::vector<std::string> contigs;
    std::vector<uint32_t> order;             // catalog position -> BED index, sorted by (contig, start)
    std::vector<int64_t> contig_off;
    std::vector<int32_t> lstart, lend;
};

Catalog build_catalog(const CallArgs &a, const std::vector<BamHeader> &hdrs)
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

// How one BAM is read against the catalog.
struct BamPlan {
    std::vector<int> cid;                            // BAM tid -> catalog contig (-1: no locus there)
    std::vector<int> tid;                            // catalog contig -> BAM tid
    std::vector<std::array<int64_t, 3>> regions;     // BAM tid, beg, end: what the .bai path fetches
    std::string bai;
    bool used_index = false;
    bool gpu_inflate = false;                        // streamed: a GPU engine inflates next to the host workers
};

BamPlan plan_bam(const std::string &path, const BamHeader &h, const Catalog &cat)
{
    BamPlan p;
    const int n_contigs = (int)cat.contigs.size();
    p.cid.assign(h.ref_names.size(), -1);
    p.tid.assign(n_contigs, -1);
    for (int c = 0; c < n_contigs; ++c) { p.tid[c] = h.tid(cat.contigs[c]); p.cid[p.tid[c]] = c; }
    // Small panels: seek through the .bai instead of inflating the whole file (SURVEY 8f rank 2).
    // Windows closer than 100 kb are fetched as one region; a read returned by two regions is kept once.
    int64_t region_span = 0, genome = 0;
    for (int64_t len : h.ref_lens) genome += len;
    for (int c = 0; c < n_contigs; ++c)
        for (int64_t i = cat.contig_off[c]; i < cat.contig_off[c + 1]; ++i) {
            const int64_t b = (int64_t)cat.lstart[i] - 10, e = (int64_t)cat.lend[i] + 10;
            if (!p.regions.empty() && p.regions.back()[0] == p.tid[c] && b <= p.regions.back()[2] + 100000) p.regions.back()[2] = std::max(p.regions.back()[2], e);
            else p.regions.push_back({(int64_t)p.tid[c], b, e});
        }
    for (const auto &r : p.regions) region_span += r[2] - r[1] + 50000;     // + typical read overhang
    p.bai = path + ".bai";
    if (!is_file(p.bai) && ends_with(path, ".bam")) p.bai = path.substr(0, path.size() - 4) + ".bai";
    const char *idx_env = getenv("INQ_BAM_INDEX");
    p.used_index = (idx_env ? atoi(idx_env) != 0 : (region_span * 10 < genome)) && is_file(p.bai);
    // BGZF blocks are inflated by the zlib-class workers AND, in runs, by a GPU engine (include/inqbgzf.h);
    // INQ_GPU_INFLATE=0 leaves it all to the workers (default: for files of 2 GB and more -- below that CUDA start-up
    // takes longer than the workers need for the file)
    const char *gi = getenv("INQ_GPU_INFLATE");
    struct stat bst;
    const bool big = stat(path.c_str(), &bst) == 0 && (uint64_t)bst.st_size >= (2ull << 30);
    p.gpu_inflate = gi ? atoi(gi) != 0 : big;
    return p;
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
    // an error of the C ABI: those the reference raises as panics exit 101, the others (no device, out of memory) 1
    void library(size_t s, int rc, const std::string &msg)
    {
        if (rc == INQ_ERR_BAD_HP || rc == INQ_ERR_BAD_SA || rc == INQ_ERR_MEDIAN_EMPTY || rc == INQ_ERR_LOCUS_START) panic(s, msg);
        else raise(s, 1, "ERROR: " + msg + " (code " + std::to_string(rc) + ")\n");
    }
};

struct SampleStats {
    bool used_index = false;
    uint64_t records = 0, pushed = 0, unpairable = 0, routed = 0, bytes_inflated = 0, bytes_inflated_gpu = 0;
    double s_wait_batch = 0, s_index = 0, s_parse = 0;     // streamed: BamReader's own split of the scan
    double s_scan = 0;
    std::chrono::steady_clock::time_point scanned;
    int slot = -1;
};

// get_phase (call.rs:349,482-491): false for the aux type the reference panics on. Phased mode reads the HP tag of
// every fetched record, whatever the filter says later. 0xFF is the ABI's "no tag"; a real value of 255 only matters
// through the HP-not-in-{0,1,2} panic of a read that passes the filter (call.rs:358), which 254 raises just the same.
bool decode_hp(bool unphased, HpType type, int64_t value, uint8_t *hp)
{
    *hp = 0xFF;
    if (unphased) return true;
    switch (type) {
    case HpType::Absent: return true;
    case HpType::U8:
    case HpType::I32: *hp = (uint8_t)value; break;          // `v as u8`
    default: return false;
    }
    if (*hp == 0xFF) *hp = 0xFE;
    return true;
}

const char *kBadHp = "Unexpected type of Aux for HP (call.rs:487)";

// One sample into a set of workers: every record goes to each worker for which htslib's fetch would return it for
// some locus, pos < end+10 && endpos > start-10 (SURVEY 8a A4), with its tid mapped to the catalog's contig; reads at
// a shard cut go to both sides. `ix` is the BAM's reader if one is open already (with its index if the plan uses one).
// Returns the message of the reference's panic on an error, empty otherwise; stops early once `abort` is set or a
// worker failed (the worker's error surfaces in take_result).
std::string scan_sample(const std::string &path, const BamPlan &plan, BamIndexedReader *ix, const std::vector<ShardWorker *> &ws,
                        int host_threads, bool unphased, SampleStats &st, const std::atomic<bool> &abort)
{
    st.used_index = plan.used_index;
    auto reaches = [&](int32_t tid, int32_t pos, int32_t end) {
        if (tid < 0 || tid >= (int32_t)plan.cid.size()) return false;
        for (const ShardWorker *w : ws)
            if (w->reaches(plan.cid[tid], pos, end)) return true;
        return false;
    };
    auto failed = [&] {
        for (ShardWorker *w : ws)
            if (w->failed()) return true;
        return false;
    };
    // a record that some worker reaches, as lite_record() classified it; false for the HP aux-type panic
    auto route = [&](const BamRecLite &r) {
        uint8_t hp;
        if (!decode_hp(unphased, r.hp_type, r.hp_value, &hp)) return false;
        // the per-read half of both filters (call.rs:297-300,350-352): such a read is skipped at every locus
        if (r.mapq <= 10 || (!unphased && hp == 0xFF)) { ++st.unpairable; return true; }
        const uint8_t fl = (uint8_t)((r.two_d ? INQ_FLAG_ACCIDENTAL_2D : 0) | (r.sa_panic ? INQ_FLAG_SA_PANIC : 0));
        const int c = plan.cid[r.tid];
        for (ShardWorker *w : ws)
            if (w->reaches(c, r.pos, r.end)) { w->add(c, r.pos, r.end, r.mapq, hp, fl, r.cigar, r.n_cigar); ++st.routed; }
        ++st.pushed;
        return true;
    };

    if (plan.used_index) {
        BamIndexedReader own;
        if (!ix) {
            if (!own.open_bam(path)) return "Error opening local BAM: " + own.error();          // call.rs:242-243
            if (!own.load_index(plan.bai)) return "Error opening BAM index: " + own.error();
            ix = &own;
        }
        std::unordered_set<uint64_t> seen;
        bool bad_hp = false;
        for (const auto &r : plan.regions) {
            if (bad_hp || abort || failed()) break;
            const bool ok = ix->fetch((int)r[0], r[1], r[2], [&](const BamRecordView &rec, uint64_t voff) {
                ++st.records;
                if (bad_hp || !seen.insert(voff).second || !reaches(rec.tid, rec.pos, rec.end)) return;
                bad_hp = !route(lite_record(rec, !unphased));
            });
            if (!ok) return "Failed to fetch region: " + ix->error();                           // call.rs:288
        }
        st.bytes_inflated = ix->bytes_inflated();
        return bad_hp ? kBadHp : "";
    }

    BamReader bam;
    if (!bam.open(path, host_threads, plan.gpu_inflate ? ws[0]->device() : -1)) return "Error opening local BAM: " + bam.error();
    RecFilter filt;
    filt.ctx = &reaches;
    filt.reach = [](const void *f, int32_t tid, int32_t pos, int32_t end) { return (*static_cast<const decltype(reaches) *>(f))(tid, pos, end); };
    filt.need_hp = !unphased;
    // two stages: this thread waits for inflated batches, walks the record boundaries and runs the parallel parse (field
    // extraction, CIGAR copy, reference length, the fetch predicate and the SA classification); a routing thread takes
    // the parsed chunks in file order (aux-type panic, routing into the workers' pinned batches, counters)
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
                    if (!route(r)) { bad_hp = true; dead = true; }
                }
            }
            if (abort || failed()) dead = true;
        }
    });
    const int parse_threads = std::max(2, host_threads / 2);     // the inflate workers own the other half of the time
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
    st.bytes_inflated_gpu = bam.gpu_bytes();
    st.s_wait_batch = bam.s_wait_batch;
    st.s_index = bam.s_index;
    st.s_parse = bam.s_parse;
    if (bad_hp) return kBadHp;
    if (!bam.error().empty()) return "Error reading BAM file: " + bam.error();
    return "";
}

// one shard's result into the sample's: concatenated in catalog order, counters summed, times of the slowest shard
void merge_result(ShardResult &acc, ShardResult &&r, size_t lo, size_t L)
{
    if (lo == 0 && r.t1.size() == L) { acc = std::move(r); return; }
    acc.t1.resize(L); acc.t2.resize(L); acc.valid.resize(L);
    std::copy(r.t1.begin(), r.t1.end(), acc.t1.begin() + lo);
    std::copy(r.t2.begin(), r.t2.end(), acc.t2.begin() + lo);
    std::copy(r.valid.begin(), r.valid.end(), acc.valid.begin() + lo);
    inq_stats &a = acc.stats;
    const inq_stats &b = r.stats;
    a.n_loci += b.n_loci; a.n_reads += b.n_reads; a.n_cigar_words += b.n_cigar_words;
    a.n_pairs += b.n_pairs; a.n_events += b.n_events; a.n_kernel_launches += b.n_kernel_launches;
    a.ms_total = std::max(a.ms_total, b.ms_total); a.ms_cigar = std::max(a.ms_cigar, b.ms_cigar); a.ms_h2d = std::max(a.ms_h2d, b.ms_h2d);
    acc.s_ctx = std::max(acc.s_ctx, r.s_ctx); acc.s_push = std::max(acc.s_push, r.s_push); acc.s_genotype = std::max(acc.s_genotype, r.s_genotype);
}

struct Run {
    const CallArgs &args;
    const std::vector<BamPlan> &plans;
    BamIndexedReader *first;                // the first BAM's reader, kept open since its header was read
    size_t L;
    int host_threads;                       // per scan
    FirstError err;
    std::vector<SampleStats> stats;
    std::vector<ShardResult> results;

    bool collect(size_t s, const std::vector<ShardWorker *> &ws)
    {
        for (ShardWorker *w : ws) {
            ShardResult r;
            if (!w->take_result(r)) { err.library(s, r.rc, r.error); return false; }
            merge_result(results[s], std::move(r), w->lo(), L);
        }
        return true;
    }

    // one set of workers: the next unstarted sample while there is one; sample k+1 is read while sample k is genotyped
    void device_loop(int slot, const std::vector<ShardWorker *> &ws, std::atomic<size_t> &next)
    {
        std::deque<size_t> pending;
        for (;;) {
            if (err.abort) break;
            const size_t s = next.fetch_add(1);
            if (s >= args.bams.size()) break;
            SampleStats &st = stats[s];
            st.slot = slot;
            const auto t0 = std::chrono::steady_clock::now();
            const std::string e = scan_sample(args.bams[s], plans[s], s == 0 ? first : nullptr, ws, host_threads, args.unphased, st, err.abort);
            st.scanned = std::chrono::steady_clock::now();
            st.s_scan = std::chrono::duration<double>(st.scanned - t0).count();
            if (!e.empty()) { err.panic(s, e); return; }
            if (err.abort) return;
            for (ShardWorker *w : ws) w->end_sample();
            pending.push_back(s);
            while (pending.size() > 1) {
                if (!collect(pending.front(), ws)) return;
                pending.pop_front();
            }
        }
        for (; !pending.empty() && !err.abort; pending.pop_front())
            if (!collect(pending.front(), ws)) return;
    }
};

// output order of `call`: -t 1 BED order (call.rs:149-157); -t > 1 sorted by (human chrom, start) (call.rs:137-145);
// one H1 / H2 column pair per sample (call.rs:101)
void write_table(const Catalog &cat, uint64_t threads, const std::vector<std::string> &names, const std::vector<ShardResult> &res)
{
    const size_t L = cat.loci.size();
    std::vector<uint32_t> pos_of(L);                 // BED index -> catalog position
    for (size_t i = 0; i < L; ++i) pos_of[cat.order[i]] = (uint32_t)i;
    std::vector<uint32_t> out_order(L);
    std::iota(out_order.begin(), out_order.end(), 0u);
    if (threads > 1)
        std::stable_sort(out_order.begin(), out_order.end(), [&](uint32_t x, uint32_t y) {
            const int c = human_compare(cat.loci[x].chrom, cat.loci[y].chrom);
            if (c != 0) return c < 0;
            return cat.loci[x].start < cat.loci[y].start;
        });
    std::string out = "chromosome\tbegin\tend";
    for (const std::string &name : names) out += "\t" + name + "_H1\t" + name + "_H2";
    out += '\n';
    for (uint32_t bi : out_order) {
        const Locus &l = cat.loci[bi];
        const uint32_t p = pos_of[bi];
        out += l.chrom;
        out += '\t';
        out += std::to_string(l.start);
        out += '\t';
        out += std::to_string(l.end);
        for (const ShardResult &r : res) {
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
}

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

int call_main(const std::vector<std::string> &argv, bool cohort, std::vector<int> devices)
{
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
    const CallArgs args = parse_call_args(argv, cohort, std::move(devices));
    const size_t S = args.bams.size();

    // every path, then every header, then the catalog against all of them (call.rs:87-90,242-243, repeats.rs:96-115),
    // then the first BAM's index: all before any record is read or any context is made
    for (const std::string &bam : args.bams) check_input(bam);
    std::vector<BamHeader> hdrs(S);
    BamIndexedReader first;
    for (size_t s = 0; s < S; ++s) {
        BamIndexedReader other;
        BamIndexedReader &ix = s ? other : first;
        if (!ix.open_bam(args.bams[s])) panic("Error opening local BAM: " + ix.error());
        hdrs[s] = ix.header();
    }
    const Catalog cat = build_catalog(args, hdrs);
    const size_t L = cat.loci.size();
    const int n_contigs = (int)cat.contigs.size();
    std::vector<BamPlan> plans;
    for (size_t s = 0; s < S; ++s) plans.push_back(plan_bam(args.bams[s], hdrs[s], cat));
    if (plans[0].used_index && !first.load_index(plans[0].bai)) panic("Error opening BAM index: " + first.error());

    // `call`: contiguous ranges of the sorted catalog, one context each, all fed by the one scan (replaces the rayon
    // fan-out of call.rs:103-145). Cuts balance the expected work: with an index, the BAM bytes its linear index places
    // around each locus (pile-up depth x read length); otherwise the locus count.
    // `call-cohort`: one context per device, at most one per sample, each with the whole catalog and scans of its own.
    const size_t n_workers = cohort ? std::min(args.devices.size(), S) : std::max<size_t>(1, std::min(args.devices.size(), std::max<size_t>(L, 1)));
    std::vector<double> weight;
    if (!cohort && plans[0].used_index && n_workers > 1) {
        weight.resize(L);
        for (int c = 0; c < n_contigs; ++c)
            for (int64_t i = cat.contig_off[c]; i < cat.contig_off[c + 1]; ++i)
                weight[i] = first.window_weight(plans[0].tid[c], (int64_t)cat.lstart[i] - 10, (int64_t)cat.lend[i] + 10);
    }
    const std::vector<size_t> cuts = balanced_cuts(L, cohort ? 1 : (int)n_workers, weight.empty() ? nullptr : weight.data());
    std::vector<std::unique_ptr<ShardWorker>> workers;
    for (size_t g = 0; g < n_workers; ++g) {
        const size_t k = cohort ? 0 : g;
        workers.emplace_back(new ShardWorker(args.devices[g], cuts[k], cuts[k + 1], n_contigs, cat.contig_off, cat.lstart.data(), cat.lend.data(),
                                             args.minlen, (uint32_t)args.support, args.unphased, n_workers <= 2 ? 4 : 2));
    }
    std::vector<std::vector<ShardWorker *>> groups(cohort ? n_workers : 1);     // the workers one scan feeds
    for (size_t g = 0; g < n_workers; ++g) groups[cohort ? g : 0].push_back(workers[g].get());

    const int total_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    Run run{args, plans, &first, L, std::max(1, total_threads / (int)groups.size())};
    run.stats.resize(S);
    run.results.resize(S);
    std::atomic<size_t> next{0};
    std::vector<std::thread> loops;
    for (size_t g = 0; g < groups.size(); ++g) loops.emplace_back([&, g] { run.device_loop((int)g, groups[g], next); });
    for (auto &t : loops) t.join();
    for (auto &w : workers) w->stop();
    if (run.err.set) {
        fputs(run.err.text.c_str(), stderr);
        return run.err.code;
    }
    const double s_flush = since(run.stats[0].scanned);

    std::vector<std::string> names;
    for (const std::string &bam : args.bams) names.push_back(args.has_sample ? args.sample_name : sample_from_path(bam));   // call.rs:91-100
    write_table(cat, args.threads, names, run.results);

    if (args.stats_json.empty()) return 0;
    FILE *f = fopen(args.stats_json.c_str(), "w");
    if (!f) return 0;
    if (!cohort) {
        const SampleStats &st = run.stats[0];
        const ShardResult &r = run.results[0];
        fprintf(f, "{\"used_index\": %d, \"records\": %" PRIu64 ", \"records_pushed\": %" PRIu64 ", \"records_unpairable\": %" PRIu64 ", \"bytes_inflated\": %" PRIu64 ", \"bytes_inflated_on_gpu\": %" PRIu64
                   ", \"n_loci\": %" PRIu64 ", \"n_reads\": %" PRIu64 ", \"n_cigar_words\": %" PRIu64 ", \"n_pairs\": %" PRIu64
                   ", \"n_events\": %" PRIu64 ", \"ms_total\": %.4f, \"ms_cigar\": %.4f, \"ms_h2d\": %.4f, \"launches\": %u"
                   ", \"n_shards\": %zu, \"records_routed\": %" PRIu64 ", \"s_ctx_create_set_loci\": %.3f, \"s_bam_scan\": %.3f, \"s_push_under_scan\": %.3f, \"s_flush_genotype\": %.3f, \"s_total\": %.3f, \"s_scan_wait_inflate\": %.3f, \"s_scan_index\": %.3f, \"s_scan_parse\": %.3f}\n",
                st.used_index ? 1 : 0, st.records, st.pushed, st.unpairable, st.bytes_inflated, st.bytes_inflated_gpu, r.stats.n_loci, r.stats.n_reads, r.stats.n_cigar_words,
                r.stats.n_pairs, r.stats.n_events, r.stats.ms_total, r.stats.ms_cigar, r.stats.ms_h2d, r.stats.n_kernel_launches, n_workers, st.routed, r.s_ctx,
                st.s_scan, r.s_push, s_flush, since(t_begin), st.s_wait_batch, st.s_index, st.s_parse);
    } else {
        double s_ctx = 0;
        for (const ShardResult &r : run.results) s_ctx = std::max(s_ctx, r.s_ctx);
        fprintf(f, "{\"n_samples\": %zu, \"n_contexts\": %zu, \"n_loci\": %zu, \"s_ctx_create_set_loci\": %.3f, \"s_total\": %.3f, \"samples\": [",
                S, n_workers, L, s_ctx, since(t_begin));
        for (size_t s = 0; s < S; ++s) {
            const SampleStats &st = run.stats[s];
            const ShardResult &r = run.results[s];
            fprintf(f, "%s{\"bam\": %s, \"context\": %d, \"used_index\": %d, \"records\": %" PRIu64 ", \"records_pushed\": %" PRIu64
                       ", \"records_unpairable\": %" PRIu64 ", \"bytes_inflated\": %" PRIu64 ", \"n_pairs\": %" PRIu64 ", \"ms_total\": %.4f"
                       ", \"s_bam_scan\": %.3f, \"s_genotype\": %.3f}",
                    s ? ", " : "", json_str(args.bams[s]).c_str(), st.slot, st.used_index ? 1 : 0, st.records, st.pushed, st.unpairable,
                    st.bytes_inflated, r.stats.n_pairs, r.stats.ms_total, st.s_scan, r.s_genotype);
        }
        fprintf(f, "]}\n");
    }
    fclose(f);
    return 0;
}

}  // namespace inqhost
