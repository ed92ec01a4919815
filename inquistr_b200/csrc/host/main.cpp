// inquistr-b200 -- C++ host of the `inquiSTR call` drop-in (the reference host is Rust; no Rust
// toolchain exists in this image, see INTEGRATION.md). Mirrors, above the C ABI of libinqcall.so:
//   CLI flags + defaults            src/main.rs:28-64
//   driver, sample name, header     src/call.rs:76-159
//   targets / validation            src/call.rs:161-202, src/repeats.rs:13-45,96-115
//   per-record fields               src/call.rs:297-299,349-352,415-459,482-491
//   ordering + row format           src/call.rs:27-65
// stdout carries only the TSV; diagnostics go to stderr. A Rust panic in the reference maps to exit
// code 101 here, `std::process::exit(1)` to 1, clap usage errors to 2.
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cinttypes>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <array>
#include <thread>
#include <unordered_set>
#include <vector>

#include "../../../include/inqcall.h"
#include "bam_reader.hpp"
#include "call_common.hpp"
#include "shard_driver.hpp"

namespace inqhost {
int combine_main(const std::vector<std::string> &files);                 // cohort_cli.cpp
int outlier_main(const std::vector<std::string> &args, int device);
int cohort_call_main(const std::vector<std::string> &args, std::vector<int> devices);   // cohort_call.cpp
}
using namespace inqhost;

namespace {

struct Args {
    std::string bam;
    bool has_region = false, has_region_file = false, has_sample = false, has_reference = false;
    std::string region, region_file, sample_name, reference;
    uint32_t minlen = 5;
    uint64_t support = 3;
    uint64_t threads = 1;
    bool unphased = false;
    std::vector<int> devices;     // extension: CUDA devices, one catalog shard + context each (also INQ_DEVICE / INQ_DEVICES)
    std::string stats_json;       // extension: timing side file
};

const char *kHelp =
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

[[noreturn]] void usage_error(const std::string &msg)
{
    fprintf(stderr, "error: %s\n\nUsage: inquistr-b200 call [OPTIONS] <BAM>\n\nFor more information, try '--help'.\n", msg.c_str());
    exit(2);
}

Args parse_args(int argc, char **argv)
{
    Args a;
    auto parse_devices = parse_device_list;
    if (const char *d = getenv("INQ_DEVICES")) { if (!parse_devices(d, &a.devices)) a.devices.clear(); }
    else if (const char *d = getenv("INQ_DEVICE")) a.devices.assign(1, atoi(d));
    if (a.devices.empty()) a.devices.assign(1, 0);
    std::vector<std::string> v(argv + 1, argv + argc);
    if (v.empty() || v[0] == "-h" || v[0] == "--help" || v[0] == "help") {
        printf("Tool to genotype STRs from long reads (B200 build of the `call` hot path)\n\n"
               "Usage: inquistr-b200 <COMMAND>\n\nCommands:\n  call         Call lengths\n"
               "  call-cohort  Call lengths in several bams against one catalog and print the combined TSV\n"
               "  combine      Combine lengths from multiple bams to a TSV\n"
               "  outlier      Find outliers from TSV\n  help         Print this message\n");
        exit(v.empty() ? 2 : 0);
    }
    if (v[0] == "-V" || v[0] == "--version") { printf("inquistr-b200 %s\n", inq_version()); exit(0); }
    if (v[0] == "bgzf-check" && v.size() >= 2) {
        // extension: own DEFLATE decoder vs zlib on every block of a BGZF file (bytes compared, MB/s of each)
        std::string rep;
        const bool ok = bgzf_selfcheck(v[1], &rep);
        printf("%s\n", rep.c_str());
        exit(ok ? 0 : 1);
    }
    if (v[0] == "baistat" && v.size() >= 2) {
        // extension: what a .bai says on its own (no BAM, no GPU): `baistat x.bam.bai [tid:beg-end]`
        BamIndexedReader ix;
        if (!ix.load_index(v[1])) { fprintf(stderr, "%s\n", ix.error().c_str()); exit(1); }
        printf("{\"refs\": %zu, \"n_no_coor\": %llu, \"mapped\": {", ix.n_refs(), (unsigned long long)ix.n_no_coor());
        bool first = true;
        for (size_t t = 0; t < ix.n_refs(); ++t)
            if (ix.n_mapped((int)t) >= 0) {
                printf("%s\"%zu\": [%lld, %lld]", first ? "" : ", ", t, (long long)ix.n_mapped((int)t), (long long)ix.n_unmapped((int)t));
                first = false;
            }
        printf("}");
        if (v.size() >= 3) {
            const size_t c1 = v[2].find(':'), c2 = v[2].find('-', c1);
            const int tid = atoi(v[2].substr(0, c1).c_str());
            const long long b = atoll(v[2].substr(c1 + 1, c2 - c1 - 1).c_str()), e = atoll(v[2].substr(c2 + 1).c_str());
            printf(", \"chunks\": [");
            first = true;
            for (const auto &c : ix.chunks_for(tid, b, e)) {
                printf("%s[%llu, %llu]", first ? "" : ", ", (unsigned long long)c.first, (unsigned long long)c.second);
                first = false;
            }
            printf("]");
        }
        printf("}\n");
        exit(0);
    }
    if (v[0] == "bamstat" && v.size() >= 2) {
        // extension: scan a BAM with the host reader only (no GPU): record counts and inflate rate;
        // `bamstat x.bam chr:beg-end` does the same through the .bai index for one region; `bamstat x.bam --parsed` runs
        // the parallel parse of the call driver instead of the sequential record walk
        if (v.size() == 3 && v[2] != "--parsed") {
            BamIndexedReader ix;
            if (!ix.open_bam(v[1]) || !ix.load_index(v[1] + ".bai")) { fprintf(stderr, "%s\n", ix.error().c_str()); exit(1); }
            const size_t c1 = v[2].find(':'), c2 = v[2].find('-', c1);
            const int tid = ix.header().tid(v[2].substr(0, c1));
            const long long b = atoll(v[2].substr(c1 + 1, c2 - c1 - 1).c_str()), e = atoll(v[2].substr(c2 + 1).c_str());
            uint64_t n = 0, words = 0;
            if (!ix.fetch(tid, b, e, [&](const BamRecordView &r, uint64_t) { ++n; words += r.n_cigar; })) { fprintf(stderr, "%s\n", ix.error().c_str()); exit(1); }
            printf("{\"records\": %llu, \"cigar_words\": %llu, \"bytes_inflated\": %llu}\n", (unsigned long long)n,
                   (unsigned long long)words, (unsigned long long)ix.bytes_inflated());
            exit(0);
        }
        BamReader rd;
        const auto t0 = std::chrono::steady_clock::now();
        int gpu = -1;                                           // `bamstat x.bam --gpu N`: GPU engine next to the workers
        if (v.size() >= 4 && v[2] == "--gpu") gpu = atoi(v[3].c_str());
        const int host_threads = (int)std::max(1u, std::thread::hardware_concurrency());
        if (!rd.open(v[1], host_threads, gpu)) { fprintf(stderr, "%s\n", rd.error().c_str()); exit(1); }
        BamRecordView r;
        uint64_t n = 0, words = 0, hp = 0, sa = 0, d2 = 0;
        if (v.size() >= 3 && v[2] == "--parsed") {
            // the host side of `call` without a device: batches parsed on the host threads exactly as the call driver
            // does it (every record kept: no catalog, phased-mode filter off), counted instead of pushed
            RecFilter filt;
            filt.reach = [](const void *, int32_t, int32_t, int32_t) { return true; };
            std::vector<ParsedChunk> chunks;
            const int parse_threads = std::max(2, host_threads / 2);
            while (rd.next_parsed(filt, parse_threads, chunks))
                for (const ParsedChunk &c : chunks) {
                    if (!c.err.empty()) { fprintf(stderr, "%s\n", c.err.c_str()); exit(1); }
                    n += c.n_records;
                    for (const BamRecLite &q : c.recs) { words += q.cigar ? q.n_cigar : 0; hp += q.hp_type != HpType::Absent; d2 += q.two_d; }
                }
            sa = d2;                                            // (the lite record only says whether the SA test came out true)
        } else {
            while (rd.next(r)) {
                ++n; words += r.n_cigar; hp += r.hp_type != HpType::Absent; sa += r.has_sa;
                bool pn = false;
                d2 += is_accidental_2d(r, &pn);
            }
        }
        if (!rd.error().empty()) { fprintf(stderr, "%s\n", rd.error().c_str()); exit(1); }
        const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        uint64_t nf = 0, nz = 0;
        inflate_counters(&nf, &nz);
        printf("{\"refs\": %zu, \"records\": %llu, \"cigar_words\": %llu, \"hp_tagged\": %llu, \"sa_tagged\": %llu, \"accidental_2d\": %llu, "
               "\"bytes_inflated\": %llu, \"seconds\": %.3f, \"inflate_GBps\": %.3f, \"blocks_fast\": %llu, \"blocks_zlib\": %llu, \"blocks_gpu\": %llu, \"bytes_gpu\": %llu}\n", rd.header().ref_names.size(),
               (unsigned long long)n, (unsigned long long)words, (unsigned long long)hp, (unsigned long long)sa, (unsigned long long)d2,
               (unsigned long long)rd.bytes_inflated(), s, rd.bytes_inflated() / 1e9 / s, (unsigned long long)nf, (unsigned long long)nz,
               (unsigned long long)rd.gpu_blocks(), (unsigned long long)rd.gpu_bytes());
        exit(0);
    }
    // cohort follow-ons of `call` (SURVEY 8f rank 3): text in, text out; cohort_cli.cpp
    if (v[0] == "combine") exit(combine_main(std::vector<std::string>(v.begin() + 1, v.end())));
    if (v[0] == "outlier") exit(outlier_main(std::vector<std::string>(v.begin() + 1, v.end()), a.devices[0]));
    // `call` over several BAMs with one context per device (cohort_call.cpp)
    if (v[0] == "call-cohort") exit(cohort_call_main(std::vector<std::string>(v.begin() + 1, v.end()), a.devices));
    if (v[0] != "call")
        usage_error("unrecognized subcommand '" + v[0] + "' (`call`, `call-cohort`, `combine` and `outlier` are implemented in this build)");
    if (v.size() == 1) { fputs(kHelp, stderr); exit(2); }                 // arg_required_else_help (main.rs:27)
    bool have_bam = false;
    auto need = [&](size_t &i, const std::string &name) -> std::string {
        if (i + 1 >= v.size()) usage_error("a value is required for '" + name + "' but none was supplied");
        return v[++i];
    };
    auto set_opt = [&](const std::string &name, const std::string &val) {
        uint64_t n = 0;
        if (name == "region") { a.region = val; a.has_region = true; }
        else if (name == "region-file") { a.region_file = val; a.has_region_file = true; }
        else if (name == "minlen") { if (!parse_u64(val, &n) || n > UINT32_MAX) usage_error("invalid value '" + val + "' for '--minlen <MINLEN>'"); a.minlen = (uint32_t)n; }
        else if (name == "support") { if (!parse_u64(val, &n)) usage_error("invalid value '" + val + "' for '--support <SUPPORT>'"); a.support = n; }
        else if (name == "threads") { if (!parse_u64(val, &n)) usage_error("invalid value '" + val + "' for '--threads <THREADS>'"); a.threads = n; }
        else if (name == "sample-name") { a.sample_name = val; a.has_sample = true; }
        else if (name == "reference") { a.reference = val; a.has_reference = true; }
        else if (name == "device") { if (!parse_u64(val, &n)) usage_error("invalid value for '--device'"); a.devices.assign(1, (int)n); }
        else if (name == "devices") { if (!parse_devices(val, &a.devices)) usage_error("invalid value '" + val + "' for '--devices <A,B,...>'"); }
        else if (name == "stats-json") a.stats_json = val;
        else usage_error("unexpected argument '--" + name + "' found");
    };
    const std::map<char, std::string> shorts = {{'r', "region"}, {'R', "region-file"}, {'m', "minlen"}, {'s', "support"}, {'t', "threads"}};
    bool only_positional = false;
    for (size_t i = 1; i < v.size(); ++i) {
        const std::string &s = v[i];
        if (!only_positional && s == "--") { only_positional = true; continue; }
        if (!only_positional && s.rfind("--", 0) == 0) {
            std::string name = s.substr(2), val;
            const size_t eq = name.find('=');
            if (name == "help") { fputs(kHelp, stdout); exit(0); }
            if (name == "unphased") { a.unphased = true; continue; }
            if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); }
            else val = need(i, "--" + name);
            set_opt(name, val);
        } else if (!only_positional && s.size() >= 2 && s[0] == '-') {
            for (size_t k = 1; k < s.size(); ++k) {
                const char c = s[k];
                if (c == 'u') { a.unphased = true; continue; }
                if (c == 'h') { fputs(kHelp, stdout); exit(0); }
                auto it = shorts.find(c);
                if (it == shorts.end()) usage_error(std::string("unexpected argument '-") + c + "' found");
                std::string val = s.substr(k + 1);
                if (!val.empty() && val[0] == '=') val = val.substr(1);
                if (val.empty()) val = need(i, std::string("-") + c);
                set_opt(it->second, val);
                break;
            }
        } else {
            if (have_bam) usage_error("unexpected argument '" + s + "' found");
            a.bam = s;
            have_bam = true;
        }
    }
    if (!have_bam) usage_error("the following required arguments were not provided:\n  <BAM>");
    return a;
}

#define INQ_CHECK(ctx, call)                                                                        \
    do {                                                                                            \
        int rc_ = (call);                                                                           \
        if (rc_ != INQ_OK) {                                                                        \
            const char *m_ = inq_last_error(ctx);                                                   \
            if (rc_ == INQ_ERR_BAD_HP || rc_ == INQ_ERR_BAD_SA || rc_ == INQ_ERR_MEDIAN_EMPTY || rc_ == INQ_ERR_LOCUS_START) \
                panic(m_);                                                                          \
            fprintf(stderr, "ERROR: %s (code %d)\n", m_, rc_);                                      \
            exit(1);                                                                                \
        }                                                                                           \
    } while (0)

}  // namespace

int main(int argc, char **argv)
{
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
    const Args args = parse_args(argc, argv);

    // call.rs:87-90
    if (!is_file(args.bam) && !starts_with(args.bam, "s3") && !starts_with(args.bam, "https://")) {
        fprintf(stderr, "ERROR: path to bam file %s is not valid!\n\n", args.bam.c_str());
        return 1;
    }
    if (!is_file(args.bam)) {
        fprintf(stderr, "ERROR: remote input (%s) is not supported by this build (no libcurl/htslib); use a local BAM\n", args.bam.c_str());
        return 1;
    }
    if (ends_with(args.bam, ".cram")) {
        fprintf(stderr, "ERROR: CRAM input is not supported by this build (no htslib CRAM codec); convert to BAM\n");
        return 1;
    }
    const std::string sample = args.has_sample ? args.sample_name : sample_from_path(args.bam);   // call.rs:91-100

    const int host_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    BamIndexedReader ibam;                                 // header now, random access later if a .bai is usable
    if (!ibam.open_bam(args.bam)) panic("Error opening local BAM: " + ibam.error());             // call.rs:242-243
    const BamHeader &hdr = ibam.header();

    // call.rs:182-202
    std::vector<Locus> loci;
    if (args.has_region && !args.has_region_file) loci.push_back(parse_region(args.region, hdr));
    else if (!args.has_region && args.has_region_file) loci = parse_bed(args.region_file, hdr);
    else {
        fprintf(stderr, "ERROR: Specify a region string (-r) or a region_file (-R)!\n\n");
        return 1;
    }
    for (const Locus &l : loci)
        if (l.start < 10) panic("attempt to subtract with overflow (locus " + l.chrom + ":" + std::to_string(l.start) + " has start < 10, call.rs:285)");
    if (args.support > UINT32_MAX) panic("support does not fit the device counter");

    // catalog sorted by (tid, start); ties keep BED order
    const size_t L = loci.size();
    std::vector<uint32_t> order(L);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
        if (loci[a].tid != loci[b].tid) return loci[a].tid < loci[b].tid;
        return loci[a].start < loci[b].start;
    });
    const int n_contigs = (int)hdr.ref_names.size();
    std::vector<int64_t> contig_off(n_contigs + 1, 0);
    std::vector<int32_t> lstart(L), lend(L), pmax(L);
    for (size_t i = 0; i < L; ++i) {
        const Locus &l = loci[order[i]];
        contig_off[l.tid + 1]++;
        lstart[i] = (int32_t)l.start;
        lend[i] = (int32_t)l.end;
    }
    for (int c = 0; c < n_contigs; ++c) contig_off[c + 1] += contig_off[c];
    for (int c = 0; c < n_contigs; ++c) {
        int32_t m = INT32_MIN;
        for (int64_t i = contig_off[c]; i < contig_off[c + 1]; ++i) { m = std::max(m, lend[i]); pmax[i] = m; }
    }

    // Small panels: seek through the .bai instead of inflating the whole file (SURVEY 8f rank 2).
    // Windows closer than 100 kb are fetched as one region; a read returned by two regions is kept once.
    std::vector<std::array<int64_t, 3>> regions;           // tid, beg, end
    int64_t region_span = 0, genome = 0;
    for (int64_t len : hdr.ref_lens) genome += len;
    for (int c = 0; c < n_contigs; ++c)
        for (int64_t i = contig_off[c]; i < contig_off[c + 1]; ++i) {
            const int64_t b = (int64_t)lstart[i] - 10, e = (int64_t)lend[i] + 10;
            if (!regions.empty() && regions.back()[0] == c && b <= regions.back()[2] + 100000) regions.back()[2] = std::max(regions.back()[2], e);
            else regions.push_back({(int64_t)c, b, e});
        }
    for (const auto &r : regions) region_span += r[2] - r[1] + 50000;     // + typical read overhang
    std::string bai = args.bam + ".bai";
    if (!is_file(bai) && ends_with(args.bam, ".bam")) bai = args.bam.substr(0, args.bam.size() - 4) + ".bai";
    const char *idx_env = getenv("INQ_BAM_INDEX");
    const bool want_index = idx_env ? atoi(idx_env) != 0 : (region_span * 10 < genome);
    const bool used_index = want_index && is_file(bai);
    if (used_index && !ibam.load_index(bai)) panic("Error opening BAM index: " + ibam.error());

    // ---- shards: contiguous ranges of the sorted catalog, one device context + host thread each (SURVEY 8e,
    // replaces the rayon fan-out of call.rs:103-145). Cuts balance the expected work: with an index, the BAM
    // bytes its linear index places around each locus (pile-up depth x read length); otherwise the locus count.
    const int n_shards = (int)std::max<size_t>(1, std::min(args.devices.size(), std::max<size_t>(L, 1)));
    std::vector<double> weight;
    if (used_index && n_shards > 1) {
        weight.resize(L);
        for (int c = 0; c < n_contigs; ++c)
            for (int64_t i = contig_off[c]; i < contig_off[c + 1]; ++i) weight[i] = ibam.window_weight(c, (int64_t)lstart[i] - 10, (int64_t)lend[i] + 10);
    }
    const std::vector<size_t> cuts = balanced_cuts(L, n_shards, weight.empty() ? nullptr : weight.data());
    const auto t_ctx0 = std::chrono::steady_clock::now();
    std::vector<std::unique_ptr<ShardWorker>> shards;
    for (int g = 0; g < n_shards; ++g)
        shards.emplace_back(new ShardWorker(args.devices[g], cuts[g], cuts[g + 1], n_contigs, contig_off, lstart.data(), lend.data(),
                                            args.minlen, (uint32_t)args.support, args.unphased, n_shards <= 2 ? 4 : 2));
    const auto t_scan0 = std::chrono::steady_clock::now();

    // one pass over the BAM; every record goes to the shards for which htslib's fetch would return it for some
    // locus: pos < end+10 && endpos > start-10 (SURVEY 8a A4). Reads at a cut are duplicated.
    uint64_t n_records = 0, n_kept = 0, n_unpairable = 0, n_routed = 0;
    std::vector<int> hit;
    // what to do with one record htslib's fetch could return for some locus
    auto consider = [&](const BamRecordView &rec) {
        if (rec.tid < 0 || rec.tid >= n_contigs) return;
        const int64_t l0 = contig_off[rec.tid], l1 = contig_off[rec.tid + 1];
        if (l0 == l1) return;
        hit.clear();
        for (int g = 0; g < n_shards; ++g)
            if (shards[g]->reaches(rec.tid, rec.pos, rec.end)) hit.push_back(g);
        if (hit.empty()) return;
        // a record the reference would fetch. Phased mode reads its HP tag first, whatever the filter says later
        // (get_phase, call.rs:349,482-491): an unexpected integer width panics for every fetched record.
        uint8_t hp = 0xFF;
        if (!args.unphased) {
            switch (rec.hp_type) {
            case HpType::Absent: break;
            case HpType::U8: hp = (uint8_t)rec.hp_value; break;
            case HpType::I32: hp = (uint8_t)rec.hp_value; break;           // `v as u8`
            default: panic("Unexpected type of Aux for HP (call.rs:487)");
            }
            // 0xFF is the ABI's "no tag"; a real value of 255 only matters through the HP-not-in-{0,1,2} panic of a
            // read that passes the filter (call.rs:358), which 254 raises just the same
            if (hp == 0xFF && rec.hp_type != HpType::Absent) hp = 0xFE;
        }
        // The per-read half of both filters (call.rs:297-300,350-352): such a read is skipped at every locus, before
        // its CIGAR or SA tag are looked at, so it is not shipped to the GPU at all.
        if (rec.mapq <= 10 || (!args.unphased && hp == 0xFF)) { ++n_unpairable; return; }
        // is_accidental_2d is only consulted on S ops of reads that passed the filter (call.rs:394): what it would
        // panic on travels as a flag and is raised by the GPU only if the read really pairs with a locus
        bool sa_panic = false;
        bool has_clip = false;
        for (uint32_t i = 0; i < rec.n_cigar && !has_clip; ++i) has_clip = (rec.cigar[i] & 0xF) == 4;
        const bool two_d = has_clip ? is_accidental_2d(rec, &sa_panic) : false;
        const uint8_t fl = (uint8_t)((two_d ? INQ_FLAG_ACCIDENTAL_2D : 0) | (sa_panic ? INQ_FLAG_SA_PANIC : 0));
        for (int g : hit) shards[g]->add(rec.tid, rec.pos, rec.end, rec.mapq, hp, fl, rec.cigar, rec.n_cigar);
        ++n_kept;
        n_routed += hit.size();
    };

    uint64_t bytes_inflated = 0, gpu_inflated = 0;
    double s_wait_batch = 0, s_index = 0, s_parse = 0;
    if (used_index) {
        std::unordered_set<uint64_t> seen;
        for (const auto &r : regions) {
            const bool ok = ibam.fetch((int)r[0], r[1], r[2], [&](const BamRecordView &rec, uint64_t voff) {
                ++n_records;
                if (seen.insert(voff).second) consider(rec);
            });
            if (!ok) panic("Failed to fetch region: " + ibam.error());       // call.rs:288
        }
        bytes_inflated = ibam.bytes_inflated();
    } else {
        BamReader bam;
        // BGZF blocks are inflated by the zlib-class workers AND, in runs, by a GPU engine on the first device
        // (include/inqbgzf.h); INQ_GPU_INFLATE=0 leaves it all to the workers
        // (default: for files of 2 GB and more -- below that CUDA start-up takes longer than the workers need for the file)
        const char *gi = getenv("INQ_GPU_INFLATE");
        struct stat bst;
        const bool big = stat(args.bam.c_str(), &bst) == 0 && (uint64_t)bst.st_size >= (2ull << 30);
        const int gpu_dev = (gi ? atoi(gi) != 0 : big) ? args.devices[0] : -1;
        if (!bam.open(args.bam, host_threads, gpu_dev)) panic("Error opening local BAM: " + bam.error());
        // records are parsed on the host threads in chunks (field extraction, CIGAR copy, reference length, the
        // fetch predicate and the SA classification run in parallel); this thread only keeps the file order: the
        // reference's aux-type panic, the routing into the shards' pinned batches and the counters
        struct ReachCtx { const std::vector<std::unique_ptr<ShardWorker>> *shards; };
        const ReachCtx rctx{&shards};
        RecFilter filt;
        filt.ctx = &rctx;
        filt.reach = [](const void *c, int32_t tid, int32_t pos, int32_t end) {
            for (const auto &sh : *static_cast<const ReachCtx *>(c)->shards)
                if (sh->reaches(tid, pos, end)) return true;
            return false;
        };
        filt.need_hp = !args.unphased;
        // two-stage consumer: this thread waits for inflated batches, walks the record boundaries and runs the parallel
        // parse; a routing thread takes the parsed chunks in file order (aux-type panic, shard routing, counters)
        std::mutex qmu;
        std::condition_variable qcv;
        std::deque<std::vector<ParsedChunk>> parsed;
        bool parse_done = false;
        std::atomic<bool> dead{false};
        auto route = [&](const std::vector<ParsedChunk> &chunks) {
            for (const ParsedChunk &pc : chunks) {
                n_records += pc.n_records;
                for (const BamRecLite &r : pc.recs) {
                    uint8_t hp = 0xFF;
                    if (!args.unphased) {                              // get_phase, call.rs:349,482-491 (see consider())
                        switch (r.hp_type) {
                        case HpType::Absent: break;
                        case HpType::U8: hp = (uint8_t)r.hp_value; break;
                        case HpType::I32: hp = (uint8_t)r.hp_value; break;
                        default: panic("Unexpected type of Aux for HP (call.rs:487)");
                        }
                        if (hp == 0xFF && r.hp_type != HpType::Absent) hp = 0xFE;
                    }
                    if (!r.cigar && r.n_cigar == 0 && (r.mapq <= 10 || (!args.unphased && hp == 0xFF))) { ++n_unpairable; continue; }
                    const uint8_t fl = (uint8_t)((r.two_d ? INQ_FLAG_ACCIDENTAL_2D : 0) | (r.sa_panic ? INQ_FLAG_SA_PANIC : 0));
                    size_t n_hit = 0;
                    for (int g = 0; g < n_shards; ++g)
                        if (shards[g]->reaches(r.tid, r.pos, r.end)) { shards[g]->add(r.tid, r.pos, r.end, r.mapq, hp, fl, r.cigar, r.n_cigar); ++n_hit; }
                    ++n_kept;
                    n_routed += n_hit;
                }
            }
            for (auto &sh : shards)
                if (sh->failed()) dead = true;                         // a shard that died (no device, out of memory) ends the scan early
        };
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
                route(chunks);
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
        if (!bam.error().empty()) panic("Error reading BAM file: " + bam.error());
        bytes_inflated = bam.bytes_inflated();
        gpu_inflated = bam.gpu_bytes();
        s_wait_batch = bam.s_wait_batch; s_index = bam.s_index; s_parse = bam.s_parse;
    }
    const double s_scan = since(t_scan0);
    const auto t_gen0 = std::chrono::steady_clock::now();

    // end of input: every shard flushes, genotypes its range (concurrently) and joins; ordered concatenation
    std::vector<std::thread> closers;
    for (auto &sh : shards) closers.emplace_back([&sh] { sh->finish(); });
    for (auto &t : closers) t.join();
    std::vector<int64_t> t1(L), t2(L);
    std::vector<uint8_t> valid(L);
    inq_stats st;
    memset(&st, 0, sizeof(st));
    double s_ctx = 0, s_push = 0;
    (void)t_ctx0;
    for (auto &sh : shards) {
        ShardResult &r = sh->result();
        if (r.rc != INQ_OK) {
            if (r.rc == INQ_ERR_BAD_HP || r.rc == INQ_ERR_BAD_SA || r.rc == INQ_ERR_MEDIAN_EMPTY || r.rc == INQ_ERR_LOCUS_START) panic(r.error);
            fprintf(stderr, "ERROR: %s (code %d)\n", r.error.c_str(), r.rc);
            return 1;
        }
        std::copy(r.t1.begin(), r.t1.end(), t1.begin() + sh->lo());
        std::copy(r.t2.begin(), r.t2.end(), t2.begin() + sh->lo());
        std::copy(r.valid.begin(), r.valid.end(), valid.begin() + sh->lo());
        st.n_loci += r.stats.n_loci; st.n_reads += r.stats.n_reads; st.n_cigar_words += r.stats.n_cigar_words;
        st.n_pairs += r.stats.n_pairs; st.n_events += r.stats.n_events; st.n_kernel_launches += r.stats.n_kernel_launches;
        st.ms_total = std::max(st.ms_total, r.stats.ms_total); st.ms_cigar = std::max(st.ms_cigar, r.stats.ms_cigar);
        st.ms_h2d = std::max(st.ms_h2d, r.stats.ms_h2d);
        s_ctx = std::max(s_ctx, r.s_ctx); s_push = std::max(s_push, r.s_push);
    }

    const double s_gen = since(t_gen0);
    // output order: -t 1 BED order (call.rs:149-157); -t > 1 sorted by (human chrom, start) (call.rs:137-145)
    std::vector<uint32_t> pos_of(L);                 // BED index -> catalog position
    for (size_t i = 0; i < L; ++i) pos_of[order[i]] = (uint32_t)i;
    std::vector<uint32_t> out_order(L);
    std::iota(out_order.begin(), out_order.end(), 0u);
    if (args.threads > 1)
        std::stable_sort(out_order.begin(), out_order.end(), [&](uint32_t a, uint32_t b) {
            const int c = human_compare(loci[a].chrom, loci[b].chrom);
            if (c != 0) return c < 0;
            return loci[a].start < loci[b].start;
        });
    std::string out;
    out.reserve(64 + L * 48);
    out += "chromosome\tbegin\tend\t" + sample + "_H1\t" + sample + "_H2\n";    // call.rs:101
    for (uint32_t bi : out_order) {
        const Locus &l = loci[bi];
        const uint32_t p = pos_of[bi];
        out += l.chrom;
        out += '\t';
        out += std::to_string(l.start);
        out += '\t';
        out += std::to_string(l.end);
        out += '\t';
        out += fmt_phase(t1[p], valid[p] & INQ_VALID_H1);
        out += '\t';
        out += fmt_phase(t2[p], valid[p] & INQ_VALID_H2);
        out += '\n';
    }
    fwrite(out.data(), 1, out.size(), stdout);
    fflush(stdout);

    if (!args.stats_json.empty()) {
        FILE *f = fopen(args.stats_json.c_str(), "w");
        if (f) {
            fprintf(f, "{\"used_index\": %d, \"records\": %" PRIu64 ", \"records_pushed\": %" PRIu64 ", \"records_unpairable\": %" PRIu64 ", \"bytes_inflated\": %" PRIu64 ", \"bytes_inflated_on_gpu\": %" PRIu64
                       ", \"n_loci\": %" PRIu64 ", \"n_reads\": %" PRIu64 ", \"n_cigar_words\": %" PRIu64 ", \"n_pairs\": %" PRIu64
                       ", \"n_events\": %" PRIu64 ", \"ms_total\": %.4f, \"ms_cigar\": %.4f, \"ms_h2d\": %.4f, \"launches\": %u"
                       ", \"n_shards\": %d, \"records_routed\": %" PRIu64 ", \"s_ctx_create_set_loci\": %.3f, \"s_bam_scan\": %.3f, \"s_push_under_scan\": %.3f, \"s_flush_genotype\": %.3f, \"s_total\": %.3f, \"s_scan_wait_inflate\": %.3f, \"s_scan_index\": %.3f, \"s_scan_parse\": %.3f}\n",
                    used_index ? 1 : 0, n_records, n_kept, n_unpairable, bytes_inflated, gpu_inflated, st.n_loci, st.n_reads, st.n_cigar_words, st.n_pairs, st.n_events,
                    st.ms_total, st.ms_cigar, st.ms_h2d, st.n_kernel_launches, n_shards, n_routed, s_ctx, s_scan, s_push, s_gen, since(t_begin), s_wait_batch, s_index, s_parse);
            fclose(f);
        }
    }
    return 0;
}
