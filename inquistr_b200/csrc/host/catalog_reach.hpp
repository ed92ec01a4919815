// catalog_reach.hpp -- the host-side rules of a locus catalog, shared by libinqcall (inq_set_loci,
// inq_push_reads_routed) and the CLI's shard workers. Plain C++17: nvcc and g++ both compile it.
//   * the fetch predicate: can a read [pos, end) reach some locus, pos < end+10 && endpos > start-10 (call.rs:285-288)
//   * the catalog checks of inq_set_loci: start >= 10, end >= start, sorted by start within each contig
// Both come from one pass over the loci, which also builds the running max of `end` per contig that the device join
// reads (DESIGN.md section 2, `pmax_end`).
#pragma once

#include <algorithm>
#include <climits>
#include <cstdint>
#include <vector>

#include "../../../include/inqcall.h"

namespace inqhost {

// what is wrong with a catalog, one bit per rule (CatalogReach::faults)
enum : unsigned { kCatStartBelow10 = 1u, kCatUnsorted = 2u, kCatEndBeforeStart = 4u };

// the error inq_set_loci reports for a catalog with these faults: end < start first, then the order, then start < 10
struct CatalogFault {
    int code;                  // INQ_OK, INQ_ERR_LOCUS_ORDER or INQ_ERR_LOCUS_START
    const char *message;       // null for INQ_OK
};
inline CatalogFault catalog_fault(unsigned faults)
{
    if (faults & kCatEndBeforeStart) return {INQ_ERR_LOCUS_ORDER, "a locus has end < start (the reference panics, repeats.rs:102-104)"};
    if (faults & kCatUnsorted) return {INQ_ERR_LOCUS_ORDER, "loci must be sorted by start within each contig"};
    if (faults & kCatStartBelow10) return {INQ_ERR_LOCUS_START, "a locus has start < 10: start-10 underflows u32 in the reference (call.rs:285)"};
    return {INQ_OK, nullptr};
}

class CatalogReach {
public:
    // (Re)build the index over loci [lo, hi) of a catalog sorted by (contig, start); contig_off are the catalog's
    // n_contigs + 1 offsets (monotonic, from 0). A slice may cut contigs; the index keeps its own copies, relative to
    // lo, in the memory of the last build (a context sets catalogs of the same size again and again). Returns faults().
    unsigned build(int32_t n_contigs, const int64_t *contig_off, const int32_t *start, const int32_t *end, int64_t lo, int64_t hi)
    {
        n_contigs_ = n_contigs;
        off_.resize((size_t)n_contigs + 1);
        start_.assign(start + lo, start + hi);
        pmax_.resize((size_t)(hi - lo));
        faults_ = 0;
        for (int32_t c = 0; c <= n_contigs; ++c) off_[c] = std::min(std::max(contig_off[c], lo), hi) - lo;
        const int32_t *e = end + lo;
        for (int32_t c = 0; c < n_contigs; ++c) {
            int32_t m = INT32_MIN, prev = INT32_MIN;      // a contig may start lower than the one before
            for (int64_t i = off_[c]; i < off_[c + 1]; ++i) {
                const int32_t s = start_[i];
                faults_ |= (s < 10 ? kCatStartBelow10 : 0u) | (s < prev ? kCatUnsorted : 0u) | (e[i] < s ? kCatEndBeforeStart : 0u);
                prev = s;
                m = std::max(m, e[i]);
                pmax_[i] = m;
            }
        }
        return faults_;
    }

    int32_t n_contigs() const { return n_contigs_; }
    const int64_t *offsets() const { return off_.data(); }     // per contig, relative to the slice
    const int32_t *pmax() const { return pmax_.data(); }       // running max of `end` within (contig, slice)
    unsigned faults() const { return faults_; }                // kCat* bits; 0 for a valid catalog

    // would htslib's fetch return a record [pos, end) on `contig` for some locus of the index? (false before a build)
    bool reaches(int32_t contig, int32_t pos, int32_t end) const
    {
        if (contig < 0 || contig >= n_contigs_) return false;
        const int64_t l0 = off_[contig], l1 = off_[contig + 1];
        if (l0 == l1) return false;
        // loci with start - 10 < endpos, and among them one with end + 10 > pos (SURVEY 8a A4)
        const int32_t *s = start_.data();
        const int64_t hi = std::lower_bound(s + l0, s + l1, (int32_t)std::min<int64_t>((int64_t)end + 10, INT32_MAX)) - s;
        return hi != l0 && (int64_t)pmax_[hi - 1] + 10 > (int64_t)pos;
    }

private:
    int32_t n_contigs_ = 0;
    std::vector<int64_t> off_;
    std::vector<int32_t> start_, pmax_;
    unsigned faults_ = 0;
};

}  // namespace inqhost
