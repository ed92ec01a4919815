// inquistr-b200 -- C++ host CLI of the `inquiSTR` drop-in: the subcommand dispatch and the extension subcommands
// `bgzf-check`, `baistat` and `bamstat`. `call` and `call-cohort` run in call_driver.cpp, `combine`, `outlier` and
// `assoc` in cohort_cli.cpp. stdout carries only the output; diagnostics go to stderr, clap usage errors exit with code 2.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/inqcall.h"
#include "bam_reader.hpp"
#include "call_common.hpp"

namespace inqhost {
int call_main(const std::vector<std::string> &args, bool cohort, std::vector<int> devices);   // call_driver.cpp
int combine_main(const std::vector<std::string> &files);                                    // cohort_cli.cpp
int outlier_main(const std::vector<std::string> &args, int device);
int assoc_main(const std::vector<std::string> &args, int device);
}
using namespace inqhost;

int main(int argc, char **argv)
{
    std::vector<int> devices;     // extension: CUDA devices (INQ_DEVICE / INQ_DEVICES, or --device / --devices)
    if (const char *d = getenv("INQ_DEVICES")) { if (!parse_device_list(d, &devices)) devices.clear(); }
    else if (const char *d = getenv("INQ_DEVICE")) devices.assign(1, atoi(d));
    if (devices.empty()) devices.assign(1, 0);
    std::vector<std::string> v(argv + 1, argv + argc);
    if (v.empty() || v[0] == "-h" || v[0] == "--help" || v[0] == "help") {
        printf("Tool to genotype STRs from long reads (B200 build of the `call` hot path)\n\n"
               "Usage: inquistr-b200 <COMMAND>\n\nCommands:\n  call         Call lengths\n"
               "  call-cohort  Call lengths in several bams against one catalog and print the combined TSV\n"
               "  combine      Combine lengths from multiple bams to a TSV\n"
               "  outlier      Find outliers from TSV\n"
               "  assoc        Test every locus of a combined TSV for association with a phenotype\n"
               "  help         Print this message\n");
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
    const std::vector<std::string> rest(v.begin() + 1, v.end());
    if (v[0] == "combine") return combine_main(rest);
    if (v[0] == "outlier") return outlier_main(rest, devices[0]);
    if (v[0] == "assoc") return assoc_main(rest, devices[0]);
    if (v[0] == "call" || v[0] == "call-cohort") return call_main(rest, v[0] == "call-cohort", devices);
    usage_error("inquistr-b200 call [OPTIONS] <BAM>",
                "unrecognized subcommand '" + v[0] + "' (`call`, `call-cohort`, `combine`, `outlier` and `assoc` are implemented in this build)");
}
