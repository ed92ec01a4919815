// call_common.hpp -- pieces of the `call` driver (main.cpp) that `call-cohort` (cohort_call.cpp) uses as they are:
// sample names, catalog parsing and validation, output order and number format.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "bam_reader.hpp"

namespace inqhost {

[[noreturn]] void panic(const std::string &msg);     // a panic in the reference: message on stderr, exit code 101
bool parse_u64(const std::string &s, uint64_t *out);
bool parse_device_list(const std::string &v, std::vector<int> *out);   // "A,B,...": 1..64 devices, each <= 1023
bool is_file(const std::string &p);
bool starts_with(const std::string &s, const char *p);
bool ends_with(const std::string &s, const char *p);
std::string sample_from_path(const std::string &path);                  // call.rs:91-100
int human_compare(const std::string &a, const std::string &b);          // human_sort 0.2.2 `compare`
std::string fmt_phase(int64_t twice, bool valid);                       // call.rs:57-65

struct Locus {
    std::string chrom;
    uint32_t start, end;
    int tid;
};
Locus new_interval(const std::string &chrom, uint64_t start64, uint64_t end64, const BamHeader &h);   // repeats.rs:96-115
Locus parse_region(const std::string &reg, const BamHeader &h);          // repeats.rs:13-29
std::vector<Locus> parse_bed(const std::string &path, const BamHeader &h);   // repeats.rs:30-45
// new_interval's message for a locus whose contig is missing from a header or too short in it
[[noreturn]] void panic_bad_contig(const std::string &chrom);

}  // namespace inqhost
