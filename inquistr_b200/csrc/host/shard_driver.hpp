// shard_driver.hpp -- multi-GPU driver of `inquistr-b200 call` (SURVEY 8e): replaces the reference's fan-out
// over loci (call.rs:103-145) with N device contexts on N host threads.
//   * the (contig, start)-sorted catalog is cut into N contiguous ranges of equal weight (weight = what the
//     caller knows about the expected work of a locus: 1, or the BAM bytes the .bai index says cover it);
//   * every record the reader yields is routed to each shard for which htslib's fetch would return it for some
//     locus of the shard (pos < end+10 && endpos > start-10, call.rs:285-288): reads at a cut go to both sides;
//   * a shard's worker thread owns one inq_ctx: it pushes full staging batches (filled directly by the reader thread,
//     which gets them before the CUDA context exists; page-locked once it does) while the reader keeps decoding, and
//     genotypes its range once the input ends;
//   * results are concatenated in shard order, which is catalog order. No collective, no device-to-device traffic.
// A device may be listed several times (one context each), which exercises the sharding on a single GPU.
// A worker may also genotype several samples in turn (`call-cohort`): end_sample() closes one sample's input, the
// worker genotypes it and clears the reads, and the reader may already fill batches of the next sample meanwhile;
// take_result() hands the samples' results back in the order they were ended. Context and catalog are set up once.
#pragma once

#include <condition_variable>
#include <cstdint>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/inqcall.h"

namespace inqhost {

// one staging batch in pinned host memory (SoA of include/inqcall.h:inq_push_reads)
struct ReadBatch {
    static constexpr size_t kWords = 32u << 20, kReads = 2u << 20;
    int32_t *contig = nullptr, *start = nullptr, *end = nullptr;
    uint64_t *off = nullptr;
    uint8_t *mapq = nullptr, *hp = nullptr, *flags = nullptr;
    uint32_t *cigar = nullptr;
    size_t n = 0, words = 0;
    void *meta_block = nullptr;
    bool room_for(size_t n_cigar) const { return n + 1 < kReads && words + n_cigar <= kWords; }
};

struct ShardResult {
    int rc = INQ_OK;
    std::string error;
    std::vector<int64_t> t1, t2;
    std::vector<uint8_t> valid;
    inq_stats stats;
    double s_ctx = 0, s_push = 0, s_genotype = 0, s_wait_input = 0;
    uint64_t reads = 0, words = 0;
};

class ShardWorker {
public:
    // catalog slice [lo, hi) of the global sorted arrays; contig_off are the GLOBAL per-contig offsets
    ShardWorker(int device, size_t lo, size_t hi, int n_contigs, const std::vector<int64_t> &contig_off,
                const int32_t *lstart, const int32_t *lend, uint32_t minlen, uint32_t support, bool unphased, int n_batches = 2);
    ~ShardWorker();
    ShardWorker(const ShardWorker &) = delete;
    ShardWorker &operator=(const ShardWorker &) = delete;

    int device() const { return device_; }
    size_t lo() const { return lo_; }
    size_t hi() const { return hi_; }
    // would htslib's fetch return a record [pos, end) on tid for some locus of this shard?
    bool reaches(int32_t tid, int32_t pos, int32_t end) const;
    // append one record to the shard's current batch (reader thread); blocks while both batches are in flight
    void add(int32_t tid, int32_t pos, int32_t end, uint8_t mapq, uint8_t hp, uint8_t flags, const uint32_t *cigar, uint32_t n_cigar);
    void finish();                       // no more input: flush, genotype, join
    ShardResult &result() { return done_.empty() ? res_ : done_.front(); }     // after finish()
    bool failed();                       // the worker hit an error (the reader may stop early)
    // per-sample cycle (reader thread): close the current sample's input; the worker genotypes it after the batches
    // added before, then clears the reads for the next sample
    void end_sample();
    // results of the ended samples, oldest first; blocks until the next one is genotyped. false if the worker failed
    // (out then carries the error)
    bool take_result(ShardResult &out);
    void stop();                         // no more samples: join the worker (no genotype of its own)

private:
    void run();
    void submit();                       // hand the current batch to the worker
    ReadBatch *take_free();

    int device_;
    size_t lo_, hi_;
    int n_contigs_;
    std::vector<int64_t> off_;           // per-contig offsets relative to lo_
    const int32_t *lstart_, *lend_;      // slice base pointers
    std::vector<int32_t> pmax_;          // running max of end within (contig, shard)
    uint32_t minlen_, support_;
    bool unphased_;

    std::thread th_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<ReadBatch *> free_, full_; // full_: a null entry marks the end of a sample
    std::vector<ReadBatch> batches_;
    ReadBatch *cur_ = nullptr;
    bool ready_ = false, done_input_ = false, failed_ = false;
    ShardResult res_;                    // the sample being pushed (or the error)
    std::deque<ShardResult> done_;       // genotyped samples not yet taken
    double s_ctx_ = 0;
};

// cut [0, L) into n contiguous ranges of (nearly) equal total weight; weight may be null (all ones)
std::vector<size_t> balanced_cuts(size_t L, int n, const double *weight);

}  // namespace inqhost
