// CatalogReach (csrc/host/catalog_reach.hpp) against brute force on seeded random catalogs and reads:
//   - reaches(): a walk over every locus of the slice on the read's contig, pos < end+10 && endpos > start-10 in 64 bits;
//   - pmax(): the running max of `end` within (contig, slice);
//   - faults() and catalog_fault(): every rule checked locus by locus, and the error inq_set_loci reports for them.
// Catalogs have empty contigs, duplicate and nested loci, slices [lo, hi) that cut contigs, and coordinates up to the
// top of the BAM range (a locus starts below 2^31-1, the longest reference a BAM header can hold); reads are on unknown
// contigs, zero-length or very long. One index is rebuilt for every catalog. Prints "bad 0 ..." with coverage counts
// when everything agrees.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>
#include "catalog_reach.hpp"

using inqhost::CatalogReach;

int main()
{
    std::mt19937_64 rng(7);
    auto uni = [&](int64_t a, int64_t b) { return a + (int64_t)(rng() % (uint64_t)(b - a + 1)); };   // [a, b]
    const int64_t kTop = INT32_MAX - 1;                     // highest locus start / read position
    uint64_t bad = 0, n_true = 0, n_false = 0, n_cut = 0, n_top = 0, n_fault[8] = {};
    CatalogReach ix;                     // rebuilt for every catalog, in the memory of the one before
    if (ix.reaches(0, 100, 200) || ix.faults()) ++bad;                                       // before the first build
    for (int trial = 0; trial < 20000; ++trial) {
        // ---- catalog
        const int n_contigs = (int)uni(0, 6);
        const bool top = trial % 3 == 0;
        const int64_t base = top ? kTop - 3000 : 10, span = top ? 3000 : uni(20, 2000);
        std::vector<int64_t> off(n_contigs + 1, 0);
        std::vector<int32_t> st, en;
        for (int c = 0; c < n_contigs; ++c) {
            const int k = uni(0, 9) < 3 ? 0 : (int)uni(1, 40);
            std::vector<std::pair<int32_t, int32_t>> loci;
            for (int j = 0; j < k; ++j) {
                if (!loci.empty() && uni(0, 9) == 0) { loci.push_back(loci.back()); continue; }          // duplicate
                const int64_t s = uni(base, std::min(base + span, kTop));
                const int r = (int)uni(0, 9);
                const int64_t len = r < 2 ? 0 : r < 7 ? uni(1, 30) : uni(100, 3000);                    // long ones nest
                loci.push_back({(int32_t)s, (int32_t)std::min(s + len, kTop)});
            }
            std::stable_sort(loci.begin(), loci.end(), [](auto &a, auto &b) { return a.first < b.first; });
            for (auto &l : loci) { st.push_back(l.first); en.push_back(l.second); }
            off[c + 1] = (int64_t)st.size();
        }
        const int64_t L = (int64_t)st.size();
        const bool faulty = L && uni(0, 3) == 0;
        if (faulty) {
            for (int m = (int)uni(1, 3); m--;) {
                const int64_t i = uni(0, L - 1);
                switch (uni(0, 2)) {
                case 0: st[i] = (int32_t)uni(-5, 9); break;
                case 1: en[i] = (int32_t)(st[i] - uni(1, 5)); break;
                default: if (i + 1 < L) std::swap(st[i], st[i + 1]);
                }
            }
        }
        int64_t lo = 0, hi = L;
        if (uni(0, 9) < 7) { lo = uni(0, L); hi = uni(lo, L); }
        std::vector<int> contig_of(L);
        for (int c = 0; c < n_contigs; ++c)
            for (int64_t i = off[c]; i < off[c + 1]; ++i) contig_of[i] = c;
        for (int c = 0; c < n_contigs; ++c) n_cut += (off[c] < lo && lo < off[c + 1]) || (off[c] < hi && hi < off[c + 1]);
        n_top += top;

        if (ix.build(n_contigs, off.data(), st.data(), en.data(), lo, hi) != ix.faults()) ++bad;

        // ---- faults and the reported error
        unsigned f = 0;
        for (int64_t i = lo; i < hi; ++i) {
            if (st[i] < 10) f |= inqhost::kCatStartBelow10;
            if (en[i] < st[i]) f |= inqhost::kCatEndBeforeStart;
            if (i > lo && contig_of[i - 1] == contig_of[i] && st[i - 1] > st[i]) f |= inqhost::kCatUnsorted;
        }
        ++n_fault[f];
        if (ix.faults() != f) ++bad;
        const inqhost::CatalogFault e = inqhost::catalog_fault(ix.faults());
        const char *want = (f & inqhost::kCatEndBeforeStart) ? "end < start" : (f & inqhost::kCatUnsorted) ? "sorted"
                           : (f & inqhost::kCatStartBelow10) ? "start < 10" : nullptr;
        const int want_code = !f ? INQ_OK : (f & (inqhost::kCatEndBeforeStart | inqhost::kCatUnsorted)) ? INQ_ERR_LOCUS_ORDER : INQ_ERR_LOCUS_START;
        if (e.code != want_code || (want ? !e.message || !strstr(e.message, want) : e.message != nullptr)) ++bad;
        if (f) continue;                 // the reach index is only defined for a valid catalog

        // ---- running max of end
        for (int64_t i = lo; i < hi; ++i) {
            int32_t m = INT32_MIN;
            for (int64_t j = std::max(lo, off[contig_of[i]]); j <= i; ++j) m = std::max(m, en[j]);
            if (ix.pmax()[i - lo] != m) ++bad;
        }

        // ---- reads
        for (int r = 0; r < 300; ++r) {
            int32_t c = (int32_t)uni(0, std::max(0, n_contigs - 1));
            const int kind = (int)uni(0, 19);
            if (kind == 0) c = -1;
            else if (kind == 1) c = n_contigs + (int32_t)uni(0, 5);
            else if (kind == 2) c = INT32_MIN;
            int64_t pos;
            if (L && uni(0, 3) != 0) {                             // near a locus edge
                const int64_t i = uni(0, L - 1);
                pos = (uni(0, 1) ? st[i] : en[i]) + uni(-40, 20);
            } else {
                pos = uni(base - 100, std::min(base + span + 100, kTop));
            }
            pos = std::min(std::max<int64_t>(pos, 0), kTop);
            const int lk = (int)uni(0, 9);
            const int64_t len = lk < 2 ? 0 : lk < 6 ? uni(1, 60) : lk < 9 ? uni(100, 20000) : uni(1000000, INT32_MAX);
            const int32_t end = (int32_t)std::min<int64_t>(pos + len, INT32_MAX);
            bool want_reach = false;
            for (int64_t i = lo; i < hi && !want_reach; ++i)
                want_reach = contig_of[i] == c && (int64_t)pos < (int64_t)en[i] + 10 && (int64_t)end > (int64_t)st[i] - 10;
            const bool got = ix.reaches(c, (int32_t)pos, end);
            if (got != want_reach) ++bad;
            (got ? n_true : n_false) += 1;
        }
    }
    printf("bad %llu reach %llu miss %llu cut %llu top %llu faults", (unsigned long long)bad, (unsigned long long)n_true,
           (unsigned long long)n_false, (unsigned long long)n_cut, (unsigned long long)n_top);
    for (unsigned f = 0; f < 8; ++f) printf(" %llu", (unsigned long long)n_fault[f]);
    printf("\n");
    return bad ? 1 : 0;
}
