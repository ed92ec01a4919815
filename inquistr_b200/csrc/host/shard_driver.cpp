// shard_driver.cpp -- see shard_driver.hpp
#include "shard_driver.hpp"
#include "../../../include/inqbgzf.h"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

namespace inqhost {

namespace {
size_t meta_bytes() { const size_t R = ReadBatch::kReads; return R * 12 + (R + 1) * 8 + R * 3 + 64; }
double now_s()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
}  // namespace

std::vector<size_t> balanced_cuts(size_t L, int n, const double *weight)
{
    std::vector<size_t> cuts(n + 1, L);
    cuts[0] = 0;
    if (n <= 1 || L == 0) return cuts;
    double total = 0;
    for (size_t i = 0; i < L; ++i) total += weight ? weight[i] : 1.0;
    double acc = 0;
    int g = 1;
    for (size_t i = 0; i < L && g < n; ++i) {
        acc += weight ? weight[i] : 1.0;
        while (g < n && acc >= total * g / n) cuts[g++] = i + 1;
    }
    for (int k = 1; k <= n; ++k) cuts[k] = std::max(cuts[k], cuts[k - 1]);
    cuts[n] = L;
    return cuts;
}

ShardWorker::ShardWorker(int device, size_t lo, size_t hi, int n_contigs, const std::vector<int64_t> &contig_off,
                         const int32_t *lstart, const int32_t *lend, uint32_t minlen, uint32_t support, bool unphased, int n_batches)
    : device_(device), lo_(lo), hi_(hi), n_contigs_(n_contigs), lstart_(lstart + lo), lend_(lend + lo), minlen_(minlen),
      support_(support), unphased_(unphased)
{
    off_.resize(n_contigs + 1);
    for (int c = 0; c <= n_contigs; ++c)
        off_[c] = (int64_t)std::min<size_t>(std::max<size_t>((size_t)contig_off[c], lo), hi) - (int64_t)lo;
    pmax_.resize(hi - lo);
    for (int c = 0; c < n_contigs; ++c) {
        int32_t m = INT32_MIN;
        for (int64_t i = off_[c]; i < off_[c + 1]; ++i) { m = std::max(m, lend_[i]); pmax_[i] = m; }
    }
    memset(&res_.stats, 0, sizeof(res_.stats));
    // staging batches: the reader fills one while others are on their way to the device (or wait for the context)
    batches_.resize((size_t)std::max(2, n_batches));
    for (ReadBatch &b : batches_) {
        const size_t R = ReadBatch::kReads;
        void *cig = nullptr, *meta = nullptr;
        if (posix_memalign(&cig, 4096, ReadBatch::kWords * 4) != 0 || posix_memalign(&meta, 4096, meta_bytes()) != 0) {
            failed_ = true;
            res_.rc = INQ_ERR_NOMEM;
            res_.error = "staging allocation failed";
            break;
        }
        b.cigar = static_cast<uint32_t *>(cig);
        b.meta_block = meta;
        uint8_t *m = static_cast<uint8_t *>(meta);
        b.off = reinterpret_cast<uint64_t *>(m); m += (R + 1) * 8;
        b.contig = reinterpret_cast<int32_t *>(m); m += R * 4;
        b.start = reinterpret_cast<int32_t *>(m); m += R * 4;
        b.end = reinterpret_cast<int32_t *>(m); m += R * 4;
        b.mapq = m; m += R;
        b.hp = m; m += R;
        b.flags = m;
        free_.push_back(&b);
    }
    th_ = std::thread([this] { run(); });
}

ShardWorker::~ShardWorker()
{
    if (th_.joinable()) {
        { std::lock_guard<std::mutex> g(mu_); done_input_ = true; }
        cv_.notify_all();
        th_.join();
    }
    for (ReadBatch &b : batches_) { free(b.cigar); free(b.meta_block); }
}

bool ShardWorker::reaches(int32_t tid, int32_t pos, int32_t end) const
{
    if (tid < 0 || tid >= n_contigs_) return false;
    const int64_t l0 = off_[tid], l1 = off_[tid + 1];
    if (l0 == l1) return false;
    // loci with start - 10 < endpos, and among them one with end + 10 > pos (SURVEY 8a A4)
    const int64_t hi = std::lower_bound(lstart_ + l0, lstart_ + l1, (int32_t)std::min<int64_t>((int64_t)end + 10, INT32_MAX)) - lstart_;
    return hi != l0 && (int64_t)pmax_[hi - 1] + 10 > (int64_t)pos;
}

bool ShardWorker::failed()
{
    std::lock_guard<std::mutex> g(mu_);
    return failed_;
}

ReadBatch *ShardWorker::take_free()
{
    std::unique_lock<std::mutex> lk(mu_);
    const double t0 = now_s();
    cv_.wait(lk, [this] { return !free_.empty() || failed_; });
    res_.s_wait_input += 0;               // (reader-side wait; the worker-side wait is accounted in run())
    (void)t0;
    if (failed_) return nullptr;
    ReadBatch *b = free_.front();
    free_.pop_front();
    b->n = 0;
    b->words = 0;
    b->off[0] = 0;
    return b;
}

void ShardWorker::submit()
{
    if (!cur_) return;
    { std::lock_guard<std::mutex> g(mu_); full_.push_back(cur_); }
    cv_.notify_all();
    cur_ = nullptr;
}

void ShardWorker::add(int32_t tid, int32_t pos, int32_t end, uint8_t mapq, uint8_t hp, uint8_t flags, const uint32_t *cigar, uint32_t n_cigar)
{
    if (cur_ && !cur_->room_for(n_cigar)) submit();
    if (!cur_) {
        cur_ = take_free();
        if (!cur_) return;                                       // worker failed: the error surfaces in finish()
    }
    if (n_cigar > ReadBatch::kWords) {                            // cannot happen with BAM (CG tag max 2^32/4 > kWords is theoretical): fail loudly
        std::lock_guard<std::mutex> g(mu_);
        failed_ = true;
        res_.rc = INQ_ERR_TOO_LARGE;
        res_.error = "a single read has more CIGAR operations than a staging batch holds";
        return;
    }
    ReadBatch &b = *cur_;
    b.contig[b.n] = tid; b.start[b.n] = pos; b.end[b.n] = end;
    b.mapq[b.n] = mapq; b.hp[b.n] = hp; b.flags[b.n] = flags;
    memcpy(b.cigar + b.words, cigar, (size_t)n_cigar * 4);
    b.words += n_cigar;
    b.off[++b.n] = b.words;
}

void ShardWorker::finish()
{
    end_sample();
    stop();
}

void ShardWorker::end_sample()
{
    submit();
    { std::lock_guard<std::mutex> g(mu_); full_.push_back(nullptr); }
    cv_.notify_all();
}

bool ShardWorker::take_result(ShardResult &out)
{
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [this] { return !done_.empty() || failed_; });
    if (done_.empty()) { out = res_; return false; }
    out = std::move(done_.front());
    done_.pop_front();
    return true;
}

void ShardWorker::stop()
{
    { std::lock_guard<std::mutex> g(mu_); done_input_ = true; }
    cv_.notify_all();
    if (th_.joinable()) th_.join();
}

void ShardWorker::run()
{
    inq_ctx *ctx = nullptr;
    auto fail = [&](int rc, const char *msg) {
        std::lock_guard<std::mutex> g(mu_);
        failed_ = true;
        if (res_.rc == INQ_OK) { res_.rc = rc; res_.error = msg ? msg : ""; }
        cv_.notify_all();
    };
    const double t0 = now_s();
    int rc = inq_ctx_create(device_, &ctx);
    if (rc != INQ_OK) { fail(rc, inq_last_error(nullptr)); return; }
    // shard view of the catalog: offsets relative to the slice, loci coordinates as they are
    rc = inq_set_loci(ctx, n_contigs_, off_.data(), lstart_, lend_);
    if (rc != INQ_OK) { fail(rc, inq_last_error(ctx)); inq_ctx_destroy(ctx); return; }
    // the staging batches were handed to the reader as ordinary memory before the context existed (CUDA start-up takes
    // 1-2 s next to the inflate threads: the reader must not wait for it); page-lock them now for the pushes
    for (ReadBatch &b : batches_) {
        inq_host_register(b.cigar, ReadBatch::kWords * 4);
        inq_host_register(b.meta_block, meta_bytes());
    }
    res_.s_ctx = s_ctx_ = now_s() - t0;

    bool need_clear = false;             // a sample has been genotyped: its reads go before the next sample's first push
    for (;;) {
        ReadBatch *b = nullptr;
        {
            std::unique_lock<std::mutex> lk(mu_);
            const double tw = now_s();
            cv_.wait(lk, [this] { return !full_.empty() || done_input_; });
            res_.s_wait_input += now_s() - tw;
            if (full_.empty()) break;
            b = full_.front();
            full_.pop_front();
        }
        if (need_clear) {
            need_clear = false;
            rc = inq_clear_reads(ctx);
            if (rc != INQ_OK) { fail(rc, inq_last_error(ctx)); break; }
        }
        if (!b) {                        // end of a sample: genotype the whole catalog against its reads
            const size_t L = hi_ - lo_;
            res_.t1.resize(L); res_.t2.resize(L); res_.valid.resize(L);
            const double tg = now_s();
            rc = inq_genotype(ctx, minlen_, support_, unphased_ ? 1 : 0, res_.t1.data(), res_.t2.data(), res_.valid.data(), &res_.stats);
            res_.s_genotype = now_s() - tg;
            if (rc != INQ_OK) { fail(rc, inq_last_error(ctx)); break; }
            {
                std::lock_guard<std::mutex> g(mu_);
                done_.push_back(std::move(res_));
                res_ = ShardResult();
                memset(&res_.stats, 0, sizeof(res_.stats));
                res_.s_ctx = s_ctx_;
            }
            cv_.notify_all();
            need_clear = true;
            continue;
        }
        const double tp = now_s();
        if (b->n) {
            rc = inq_push_reads(ctx, b->n, b->contig, b->start, b->end, b->mapq, b->hp, b->flags, b->off, b->cigar);
            res_.reads += b->n;
            res_.words += b->words;
        }
        res_.s_push += now_s() - tp;
        if (rc != INQ_OK) { fail(rc, inq_last_error(ctx)); break; }
        { std::lock_guard<std::mutex> g(mu_); free_.push_back(b); }
        cv_.notify_all();
    }
    for (ReadBatch &b : batches_) { inq_host_unregister(b.cigar); inq_host_unregister(b.meta_block); }
    inq_ctx_destroy(ctx);
}

}  // namespace inqhost
