// call_common.cpp -- see call_common.hpp
#include "call_common.hpp"

#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>

#include <sys/stat.h>

namespace inqhost {

void panic(const std::string &msg)
{
    // a panic in the reference: message on stderr, exit code 101
    fprintf(stderr, "thread 'main' panicked: %s\n", msg.c_str());
    exit(101);
}

void usage_error(const std::string &usage, const std::string &msg)
{
    fprintf(stderr, "error: %s\n\nUsage: %s\n\nFor more information, try '--help'.\n", msg.c_str(), usage.c_str());
    exit(2);
}

bool parse_u64(const std::string &s, uint64_t *out)
{
    if (s.empty()) return false;
    uint64_t v = 0;
    for (char c : s) {
        if (c < '0' || c > '9') return false;
        if (v > (UINT64_MAX - (uint64_t)(c - '0')) / 10) return false;
        v = v * 10 + (uint64_t)(c - '0');
    }
    *out = v;
    return true;
}

bool parse_device_list(const std::string &v, std::vector<int> *out)
{
    out->clear();
    size_t p0 = 0;
    while (p0 <= v.size()) {
        size_t p1 = v.find(',', p0);
        if (p1 == std::string::npos) p1 = v.size();
        uint64_t n = 0;
        if (!parse_u64(v.substr(p0, p1 - p0), &n) || n > 1023) return false;
        out->push_back((int)n);
        p0 = p1 + 1;
    }
    return !out->empty() && out->size() <= 64;
}

bool is_file(const std::string &p)
{
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode);
}
bool starts_with(const std::string &s, const char *p) { return s.rfind(p, 0) == 0; }
bool ends_with(const std::string &s, const char *p)
{
    const size_t n = strlen(p);
    return s.size() >= n && s.compare(s.size() - n, n, p) == 0;
}
static void replace_all(std::string &s, const std::string &from, const std::string &to)
{
    for (size_t p = 0; (p = s.find(from, p)) != std::string::npos; p += to.size()) s.replace(p, from.size(), to);
}

// call.rs:91-100: PathBuf::file_stem then .replace(".bam","").replace(".cram","")
std::string sample_from_path(const std::string &path)
{
    size_t slash = path.find_last_of('/');
    std::string name = slash == std::string::npos ? path : path.substr(slash + 1);
    size_t dot = name.find_last_of('.');
    if (dot != std::string::npos && dot != 0) name = name.substr(0, dot);
    replace_all(name, ".bam", "");
    replace_all(name, ".cram", "");
    return name;
}

// human_sort 0.2.2 `compare` (Cargo.lock dependency; published algorithm restated): numeric runs
// compare as u32 numbers, other chars compare individually, exhaustion falls back to string order.
int human_compare(const std::string &a, const std::string &b)
{
    size_t i = 0, j = 0;
    while (i < a.size() && j < b.size()) {
        const bool da = a[i] >= '0' && a[i] <= '9', db = b[j] >= '0' && b[j] <= '9';
        if (da && db) {
            uint32_t x = 0, y = 0;
            while (i < a.size() && a[i] >= '0' && a[i] <= '9') x = x * 10u + (uint32_t)(a[i++] - '0');
            while (j < b.size() && b[j] >= '0' && b[j] <= '9') y = y * 10u + (uint32_t)(b[j++] - '0');
            if (x != y) return x < y ? -1 : 1;
        } else {
            const unsigned char ca = (unsigned char)a[i], cb = (unsigned char)b[j];
            if (ca != cb) return ca < cb ? -1 : 1;
            ++i;
            ++j;
        }
    }
    const int c = a.compare(b);
    return (c > 0) - (c < 0);
}

// Rust `{}` of an f64 that is NaN or a multiple of 0.5 (call.rs:57-65)
std::string fmt_phase(int64_t twice, bool valid)
{
    if (!valid) return "NaN";
    char buf[64];
    if ((twice & 1) == 0) snprintf(buf, sizeof(buf), "%" PRId64, twice / 2);
    else if (twice == -1) snprintf(buf, sizeof(buf), "-0.5");
    else snprintf(buf, sizeof(buf), "%" PRId64 ".5", twice / 2);
    return buf;
}

void panic_bad_contig(const std::string &chrom)
{
    panic("Chromosome " + chrom + " is not in the fasta file or the end coordinate is out of bounds");
}

// repeats.rs:96-115
Locus new_interval(const std::string &chrom, uint64_t start64, uint64_t end64, const BamHeader &h)
{
    if (start64 > UINT32_MAX || end64 > UINT32_MAX) panic("called `Result::unwrap()` on an `Err` value: TryFromIntError(())");   // repeats.rs:91-92
    const uint32_t start = (uint32_t)start64, end = (uint32_t)end64;
    if (end < start)
        panic("End coordinate is smaller than start coordinate for " + chrom + ":" + std::to_string(start) + "-" + std::to_string(end));
    const int tid = h.tid(chrom);
    if (tid >= 0 && (int64_t)end < h.ref_lens[tid]) return Locus{chrom, start, end, tid};
    panic_bad_contig(chrom);
}

// repeats.rs:13-29: split(':')[0], split(':')[1].split('-')[0..1], parse::<u32>
Locus parse_region(const std::string &reg, const BamHeader &h)
{
    const size_t colon = reg.find(':');
    if (colon == std::string::npos) panic("index out of bounds: the len is 1 but the index is 1");
    const std::string chrom = reg.substr(0, colon);
    std::string interval = reg.substr(colon + 1);
    const size_t colon2 = interval.find(':');
    if (colon2 != std::string::npos) interval = interval.substr(0, colon2);
    const size_t dash = interval.find('-');
    if (dash == std::string::npos) panic("index out of bounds: the len is 1 but the index is 1");
    std::string s0 = interval.substr(0, dash), s1 = interval.substr(dash + 1);
    const size_t dash2 = s1.find('-');
    if (dash2 != std::string::npos) s1 = s1.substr(0, dash2);
    uint64_t a = 0, b = 0;
    auto parse_u32 = [](std::string s, uint64_t *out) {        // Rust's u32::from_str accepts a leading '+'
        if (!s.empty() && s[0] == '+') s = s.substr(1);
        return parse_u64(s, out) && *out <= UINT32_MAX;
    };
    if (!parse_u32(s0, &a) || !parse_u32(s1, &b)) panic("called `Result::unwrap()` on an `Err` value: ParseIntError { kind: InvalidDigit }");
    return new_interval(chrom, a, b, h);
}

// repeats.rs:30-45 via bio::io::bed::Reader (csv: tab separated, no header, '#' comments)
std::vector<Locus> parse_bed(const std::string &path, const BamHeader &h)
{
    std::ifstream in(path);
    if (!in) panic("Problem reading bed file!: Os { code: 2, kind: NotFound, message: \"No such file or directory\" }");
    std::vector<Locus> out;
    std::string line;
    while (std::getline(in, line)) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (line.empty() || line[0] == '#') continue;
        std::vector<std::string> f;
        size_t a = 0;
        while (f.size() < 3) {
            size_t b = line.find('\t', a);
            if (b == std::string::npos) { f.push_back(line.substr(a)); break; }
            f.push_back(line.substr(a, b - a));
            a = b + 1;
        }
        uint64_t s = 0, e = 0;
        if (f.size() < 3 || !parse_u64(f[1], &s) || !parse_u64(f[2], &e)) panic("Error reading bed record.: " + line);
        out.push_back(new_interval(f[0], s, e, h));
    }
    return out;
}

}  // namespace inqhost
