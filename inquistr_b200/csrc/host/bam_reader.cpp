// bam_reader.cpp -- see bam_reader.hpp. SAM/BAM spec v1 section 4 (BGZF 4.1, BAM 4.2).
#include "bam_reader.hpp"
#include "crc32_fast.hpp"
#include "inflate_fast.hpp"
#include "../../../include/inqbgzf.h"
#include "../../../include/inqcall.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <thread>

namespace inqhost {

namespace {

inline uint16_t rd16(const uint8_t *p) { return (uint16_t)(p[0] | (p[1] << 8)); }
inline uint32_t rd32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline int32_t rdi32(const uint8_t *p) { return (int32_t)rd32(p); }

std::atomic<uint64_t> g_fast_blocks{0}, g_zlib_blocks{0};

bool inflate_block(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len, uint32_t crc)
{
    if (out_len == 0) return true;
    // own one-shot decoder first (inflate_fast.hpp); zlib when it declines or the CRC disagrees
    thread_local FastInflater fi;
    if (fi.inflate(in, in_len, out, out_len) && crc32_buffer(out, out_len) == crc) {
        g_fast_blocks.fetch_add(1, std::memory_order_relaxed);
        return true;
    }
    g_zlib_blocks.fetch_add(1, std::memory_order_relaxed);
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    zs.next_in = const_cast<Bytef *>(in);
    zs.avail_in = (uInt)in_len;
    zs.next_out = out;
    zs.avail_out = (uInt)out_len;
    int rc = inflate(&zs, Z_FINISH);
    inflateEnd(&zs);
    if (rc != Z_STREAM_END || zs.total_out != out_len) return false;
    return crc32_buffer(out, out_len) == crc;
}

}  // namespace

void inflate_counters(uint64_t *fast, uint64_t *zlib_fallback)
{
    *fast = g_fast_blocks.load();
    *zlib_fallback = g_zlib_blocks.load();
}

// single-threaded differential check + timing of the two decoders on every block of a BGZF file
bool bgzf_selfcheck(const std::string &path, std::string *report)
{
    FILE *fp = fopen(path.c_str(), "rb");
    if (!fp) { *report = "cannot open " + path; return false; }
    std::vector<uint8_t> file;
    uint8_t buf[1 << 16];
    size_t k;
    while ((k = fread(buf, 1, sizeof(buf), fp)) > 0) file.insert(file.end(), buf, buf + k);
    fclose(fp);
    file.resize(file.size() + 16);
    size_t p = 0, blocks = 0, mism = 0, declined = 0;
    uint64_t out_bytes = 0;
    double t_fast = 0, t_zlib = 0, t_crc = 0, t_crcf = 0;
    FastInflater fi;
    std::vector<uint8_t> a(1 << 16), b(1 << 16);
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    while (p + 28 <= file.size() - 16) {
        const uint16_t xlen = rd16(&file[p + 10]);
        const size_t bsize = (size_t)rd16(&file[p + 16]) + 1;
        // a BGZF member: gzip magic, deflate, FEXTRA, the 6-byte 'BC' subfield first (what every BGZF writer emits)
        if (file[p] != 0x1f || file[p + 1] != 0x8b || file[p + 2] != 8 || !(file[p + 3] & 4) || file[p + 12] != 'B' || file[p + 13] != 'C' ||
            bsize < (size_t)12 + xlen + 8 || p + bsize > file.size() - 16) {
            *report = "not a BGZF member at offset " + std::to_string(p);
            return false;
        }
        const uint8_t *pay = &file[p + 12 + xlen];
        const size_t in_len = bsize - 12 - xlen - 8;
        const uint32_t crc = rd32(&file[p + bsize - 8]), isize = rd32(&file[p + bsize - 4]);
        if (isize) {
            double t0 = now();
            const bool okf = fi.inflate(pay, in_len, a.data(), isize);
            t_fast += now() - t0;
            t0 = now();
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            inflateInit2(&zs, -15);
            zs.next_in = const_cast<Bytef *>(pay); zs.avail_in = (uInt)in_len; zs.next_out = b.data(); zs.avail_out = isize;
            const int rc = inflate(&zs, Z_FINISH);
            inflateEnd(&zs);
            t_zlib += now() - t0;
            t0 = now();
            const bool crc_ok = crc32(crc32(0L, Z_NULL, 0), b.data(), isize) == crc;
            t_crc += now() - t0;
            t0 = now();
            const bool crc_same = crc32_buffer(b.data(), isize) == crc;
            t_crcf += now() - t0;
            if (crc_ok != crc_same) ++mism;
            if (rc != Z_STREAM_END || !crc_ok) ++mism;
            else if (!okf) ++declined;
            else if (memcmp(a.data(), b.data(), isize) != 0) ++mism;
            out_bytes += isize;
        }
        ++blocks;
        p += bsize;
    }
    char line[512];
    snprintf(line, sizeof(line), "{\"blocks\": %zu, \"bytes\": %llu, \"mismatch\": %zu, \"fast_declined\": %zu, \"fast_MBps\": %.1f, \"zlib_MBps\": %.1f, \"crc_MBps\": %.1f, \"crc_clmul_MBps\": %.1f}",
             blocks, (unsigned long long)out_bytes, mism, declined, out_bytes / 1e6 / t_fast, out_bytes / 1e6 / t_zlib, out_bytes / 1e6 / t_crc, out_bytes / 1e6 / t_crcf);
    *report = line;
    return mism == 0;
}

int BamHeader::tid(const std::string &name) const
{
    for (size_t i = 0; i < ref_names.size(); ++i)
        if (ref_names[i] == name) return (int)i;
    return -1;
}

BamReader::HostBuf BamReader::alloc_buf(size_t cap)
{
    HostBuf b;
    void *p = nullptr;
    if (posix_memalign(&p, 2u << 20, cap) != 0) return b;
    madvise(p, cap, MADV_HUGEPAGE);                              // fewer first-touch faults while 16 workers write into it
    b.p = static_cast<uint8_t *>(p);
    b.cap = cap;
    return b;
}

void BamReader::free_buf(HostBuf &b)
{
    if (!b.p) return;
    if (b.registered) inq_host_unregister(b.p);
    free(b.p);
    b = HostBuf();
}

BamReader::~BamReader()
{
    {
        std::lock_guard<std::mutex> lk(mu_);
        stop_ = true;
    }
    cv_.notify_all();
    cv_work_.notify_all();
    if (producer_.joinable()) producer_.join();
    for (auto &t : workers_) t.join();
    for (auto &t : gpu_threads_) t.join();
    for (auto &q : queue_) free_buf(q->data);
    for (auto &b : pool_) free_buf(b.data);
    if (cur_batch_) free_buf(cur_batch_->data);
    if (map_) munmap(const_cast<uint8_t *>(map_), map_len_);
    if (fd_ >= 0) close(fd_);
}

bool BamReader::open(const std::string &path, int threads, int gpu_device)
{
    threads_ = std::max(1, threads);
    gpu_device_ = gpu_device;
    fd_ = ::open(path.c_str(), O_RDONLY);
    if (fd_ < 0) { err_ = "cannot open " + path; return false; }
    struct stat st;
    if (fstat(fd_, &st) != 0) { err_ = "cannot stat " + path; return false; }
    map_len_ = (size_t)st.st_size;
    if (map_len_) {
        void *m = mmap(nullptr, map_len_, PROT_READ, MAP_SHARED, fd_, 0);
        if (m == MAP_FAILED) { err_ = "cannot map " + path; return false; }
        map_ = static_cast<const uint8_t *>(m);
        madvise(m, map_len_, MADV_SEQUENTIAL);
    }
    cur_batch_.reset(new Batch());
    producer_ = std::thread(&BamReader::producer, this);
    for (int t = 0; t < threads_; ++t) workers_.emplace_back(&BamReader::inflater, this);
    if (gpu_device_ >= 0)
        for (int g = 0; g < kGpuEngines; ++g) gpu_threads_.emplace_back(&BamReader::gpu_inflater, this);
    return parse_header();
}

// one batch of BGZF blocks: the file is memory-mapped, so the I/O thread only walks the block headers (two cache lines
// per block); the inflaters read the compressed payloads straight from the page cache, nothing is copied on the host
bool BamReader::read_batch(Batch &out)
{
    {
        std::lock_guard<std::mutex> lk(mu_);
        if (!pool_.empty()) { out.data = pool_.back().data; pool_.pop_back(); }
    }
    if (out.data.empty()) out.data = alloc_buf(kSlack + kOutCap);
    if (out.data.empty()) { out.err = "out of memory"; return false; }
    out.comp.p = const_cast<uint8_t *>(map_);                   // (not owned: BlockRef::in_off is an offset into the mapping)
    out.comp.cap = map_len_;
    size_t p = map_pos_, out_total = 0;
    const uint8_t *comp = map_;
    while (out.blocks.size() < kMaxBlocks && p < map_len_) {
        if (map_len_ - p < 18) { out.err = "truncated BGZF block"; return false; }
        const uint8_t *h = comp + p;
        if (h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) { out.err = "not a BGZF block (bad gzip header)"; return false; }
        const uint16_t xlen = rd16(h + 10);
        if (map_len_ - p < 12u + xlen) { out.err = "truncated BGZF extra field"; return false; }
        int bsize = -1;
        for (size_t i = 0; i + 4 <= xlen;) {
            const uint16_t slen = rd16(h + 12 + i + 2);
            if (h[12 + i] == 'B' && h[12 + i + 1] == 'C' && slen == 2 && i + 6 <= xlen) bsize = rd16(h + 12 + i + 4);
            i += 4 + slen;
        }
        if (bsize < 0) { out.err = "BGZF block without BC subfield"; return false; }
        const size_t total = (size_t)bsize + 1;
        if (total < 12u + xlen + 8u) { out.err = "corrupt BGZF block size"; return false; }
        if (map_len_ - p < total) { out.err = "truncated BGZF block"; return false; }
        BlockRef b;
        b.in_off = p + 12 + xlen;
        b.in_len = total - 12 - xlen - 8;
        b.crc = rd32(comp + p + total - 8);
        b.out_len = rd32(comp + p + total - 4);
        if (b.out_len > 65536) { out.err = "BGZF block larger than 64 KB"; return false; }
        if (out_total + b.out_len > kOutCap) break;
        b.out_off = out_total;
        out_total += b.out_len;
        out.blocks.push_back(b);
        p += total;
    }
    map_pos_ = p;
    if (p >= map_len_) out.eof = true;
    out.size = kSlack + out_total;
    return true;
}

void BamReader::producer()
{
    for (;;) {
        std::unique_ptr<Batch> b(new Batch());
        const bool ok = read_batch(*b);
        if (!ok) { b->bad = true; b->blocks.clear(); }
        const bool last = !ok || b->eof;
        {
            std::unique_lock<std::mutex> lk(mu_);
            cv_.wait(lk, [&] { return stop_ || queue_.size() < kInFlight; });
            if (stop_) { free_buf(b->data); return; }
            queue_.push_back(std::move(b));
            if (last) producer_done_ = true;
        }
        cv_work_.notify_all();
        cv_.notify_all();
        if (last) return;
    }
}

// worker: CRC32 of blocks the GPU inflated first (they gate the batch), then the next block of the oldest batch that
// still has blocks to hand out
void BamReader::inflater()
{
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
        Batch *b = nullptr;
        size_t i = 0;
        bool crc_only = false;
        while (!crc_.empty() && crc_.front().next >= crc_.front().end) crc_.pop_front();
        if (!crc_.empty()) {
            b = crc_.front().b;
            i = crc_.front().next++;
            crc_only = true;
        } else {
            for (auto &q : queue_)
                if (q->next_block < q->blocks.size()) { b = q.get(); i = q->next_block++; break; }
        }
        if (!b) {
            if (stop_) return;
            if (producer_done_) {
                bool pending = false;
                for (auto &q : queue_) pending = pending || q->done_blocks < q->blocks.size();
                if (!pending) return;
            }
            cv_work_.wait(lk);
            continue;
        }
        lk.unlock();
        const BlockRef &r = b->blocks[i];
        uint8_t *dst = b->data.data() + kSlack + r.out_off;
        bool ok;
        if (crc_only) {
            ok = r.out_len == 0 || crc32_buffer(dst, r.out_len) == r.crc;
            if (!ok) ok = inflate_block(b->comp.data() + r.in_off, r.in_len, dst, r.out_len, r.crc);   // the device got it wrong: redo here
        } else {
            ok = inflate_block(b->comp.data() + r.in_off, r.in_len, dst, r.out_len, r.crc);
        }
        lk.lock();
        if (!ok) { b->bad = true; if (b->err.empty()) b->err = "BGZF inflate / CRC failure"; }
        if (++b->done_blocks == b->blocks.size()) cv_.notify_all();
    }
}

// GPU engine thread: claims runs of consecutive blocks of the oldest batch, inflates them on the device
// (include/inqbgzf.h) and queues their CRC checks for the workers. Blocks the kernel declines are inflated here.
void BamReader::gpu_inflater()
{
    constexpr size_t kRun = 1024, kMinRun = 48;
    inq_bgzf_engine *eng = nullptr;
    constexpr size_t kStage = kRun * (65536 + 64);
    if (inq_bgzf_engine_create(gpu_device_, kStage, kOutCap, (uint32_t)kRun, &eng) != INQ_OK) return;   // no device: the workers do it all
    void *stage_v = nullptr;
    if (inq_host_alloc(kStage + 64, &stage_v) != INQ_OK) { inq_bgzf_engine_destroy(eng); return; }
    uint8_t *stage = static_cast<uint8_t *>(stage_v);
    std::vector<inq_zblock> desc(kRun);
    std::vector<uint32_t> status(kRun);
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
        Batch *b = nullptr;
        size_t a = 0, e = 0;
        // newest batch first: the workers drain the oldest one, the device works ahead of them
        for (auto it = queue_.rbegin(); it != queue_.rend(); ++it) {
            auto &q = *it;
            if (q->blocks.size() - q->next_block >= kMinRun) {
                b = q.get();
                a = q->next_block;
                e = std::min(q->blocks.size(), a + kRun);
                q->next_block = e;
                break;
            }
        }
        if (!b) {
            if (stop_) break;
            if (producer_done_) {
                bool pending = false;
                for (auto &q : queue_) pending = pending || q->blocks.size() - q->next_block >= kMinRun;
                if (!pending) break;
            }
            cv_work_.wait(lk);
            continue;
        }
        lk.unlock();
        // page-lock the batch's output buffer the first time it is seen (buffers are recycled: a few times only); the
        // compressed bytes of the run go from the page cache into this thread's page-locked staging buffer
        if (!b->data.registered) b->data.registered = inq_host_register(b->data.data(), b->data.cap) == INQ_OK;
        uint64_t bytes = 0;
        const size_t in_lo = b->blocks[a].in_off & ~(size_t)7, in_hi = b->blocks[e - 1].in_off + b->blocks[e - 1].in_len;
        if (in_hi - in_lo > kStage) {                             // cannot happen with <= 64 KB blocks and kRun of them; be safe
            lk.lock();
            b->next_block = a;                                    // hand the run back to the workers
            cv_work_.notify_all();
            break;
        }
        memcpy(stage, b->comp.data() + in_lo, in_hi - in_lo);
        for (size_t i = a; i < e; ++i) {
            const BlockRef &r = b->blocks[i];
            desc[i - a] = inq_zblock{(uint64_t)(r.in_off - in_lo), (uint64_t)(kSlack + r.out_off), (uint32_t)r.in_len, (uint32_t)r.out_len};
            bytes += r.out_len;
        }
        const int rc = inq_bgzf_engine_run(eng, stage, in_hi - in_lo, desc.data(), (uint32_t)(e - a), b->data.data(), status.data(), nullptr);
        bool bad = false;
        for (size_t i = a; i < e; ++i)
            if (rc != INQ_OK || status[i - a] != 0) {
                const BlockRef &r = b->blocks[i];
                if (!inflate_block(b->comp.data() + r.in_off, r.in_len, b->data.data() + kSlack + r.out_off, r.out_len, r.crc)) bad = true;
            }
        gpu_blocks_.fetch_add(e - a, std::memory_order_relaxed);
        gpu_bytes_.fetch_add(bytes, std::memory_order_relaxed);
        lk.lock();
        if (bad) { b->bad = true; if (b->err.empty()) b->err = "BGZF inflate / CRC failure"; }
        crc_.push_back(CrcRange{b, a, e});
        cv_work_.notify_all();
    }
    lk.unlock();
    inq_host_free(stage);
    inq_bgzf_engine_destroy(eng);
}

// make the next batch current, keeping the unconsumed tail of the old one in front of it
bool BamReader::next_batch()
{
    if (eof_) return false;
    std::unique_ptr<Batch> nb;
    {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !queue_.empty() && queue_.front()->done_blocks == queue_.front()->blocks.size(); });
        nb = std::move(queue_.front());
        queue_.pop_front();
    }
    cv_.notify_all();
    if (nb->bad || !nb->err.empty()) {
        err_ = nb->err.empty() ? "BGZF read failure" : nb->err;
        eof_ = true;
        free_buf(nb->data);
        return false;
    }
    const size_t tail = end_ - cur_;
    const size_t payload = nb->size - kSlack;
    total_out_ += payload;
    if (nb->eof) eof_ = true;
    if (tail <= kSlack) {
        if (tail) memcpy(nb->data.data() + kSlack - tail, cur_batch_->data.data() + cur_, tail);
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (!cur_batch_->data.empty()) {
                if (pool_.size() < kInFlight + 3) pool_.push_back(Buffers{cur_batch_->data, HostBuf()});
                else free_buf(cur_batch_->data);
            }
        }
        cur_batch_ = std::move(nb);
        cur_ = kSlack - tail;
        end_ = cur_batch_->size;
    } else {                                        // a record larger than the slack: concatenate into a one-off buffer
        HostBuf joined = alloc_buf(kSlack + tail + payload + 64);
        if (joined.empty()) { err_ = "out of memory"; eof_ = true; return false; }
        memcpy(joined.data() + kSlack, cur_batch_->data.data() + cur_, tail);
        memcpy(joined.data() + kSlack + tail, nb->data.data() + kSlack, payload);
        const bool was_eof = nb->eof;
        free_buf(cur_batch_->data);
        free_buf(nb->data);
        cur_batch_.reset(new Batch());
        cur_batch_->data = joined;
        cur_batch_->size = kSlack + tail + payload;
        cur_batch_->eof = was_eof;
        cur_ = kSlack;
        end_ = cur_batch_->size;
    }
    return payload > 0 || !eof_;
}

bool BamReader::ensure_bytes(size_t n)
{
    while (end_ - cur_ < n) {
        if (eof_) return false;
        next_batch();
        if (!err_.empty()) return false;
    }
    return true;
}

bool BamReader::parse_header()
{
    if (!ensure_bytes(12) || memcmp(cur_batch_->data.data() + cur_, "BAM\1", 4) != 0) { if (err_.empty()) err_ = "not a BAM file (bad magic)"; return false; }
    const uint32_t l_text = rd32(cur_batch_->data.data() + cur_ + 4);
    cur_ += 8;
    if (!ensure_bytes((size_t)l_text + 4)) { if (err_.empty()) err_ = "truncated BAM header text"; return false; }
    header_.text.assign((const char *)cur_batch_->data.data() + cur_, l_text);
    cur_ += l_text;
    const uint32_t n_ref = rd32(cur_batch_->data.data() + cur_);
    cur_ += 4;
    for (uint32_t i = 0; i < n_ref; ++i) {
        if (!ensure_bytes(4)) { if (err_.empty()) err_ = "truncated BAM reference list"; return false; }
        const uint32_t l_name = rd32(cur_batch_->data.data() + cur_);
        cur_ += 4;
        if (!ensure_bytes((size_t)l_name + 4)) { if (err_.empty()) err_ = "truncated BAM reference list"; return false; }
        std::string name((const char *)cur_batch_->data.data() + cur_, l_name);
        if (!name.empty() && name.back() == '\0') name.pop_back();
        cur_ += l_name;
        header_.ref_names.push_back(name);
        header_.ref_lens.push_back((int64_t)rd32(cur_batch_->data.data() + cur_));
        cur_ += 4;
    }
    return true;
}

bool BamReader::next(BamRecordView &rec)
{
    if (!ensure_bytes(4)) {
        if (err_.empty() && end_ != cur_) err_ = "truncated BAM record";
        return false;
    }
    const uint32_t block_size = rd32(cur_batch_->data.data() + cur_);
    if (block_size < 32) { err_ = "corrupt BAM record"; return false; }
    if (!ensure_bytes((size_t)block_size + 4)) { if (err_.empty()) err_ = "truncated BAM record"; return false; }
    const uint8_t *p = cur_batch_->data.data() + cur_ + 4;       // record body, parsed in place
    cur_ += (size_t)block_size + 4;
    return parse_bam_record(p, block_size, rec, cg_, err_);
}

bool BamReader::next_parsed(const RecFilter &filter, int parse_threads, std::vector<ParsedChunk> &chunks)
{
    chunks.clear();
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = now();
    double t_waited = 0;
    // 1. record boundaries of what is inflated and contiguous right now (one 4-byte hop per record)
    std::vector<std::pair<size_t, uint32_t>> recs;               // offset of the record body, block_size
    for (;;) {
        if (end_ - cur_ < 4) {
            if (!recs.empty()) break;
            const double tw = now();
            const bool okb = ensure_bytes(4);
            t_waited += now() - tw;
            if (!okb) {
                if (err_.empty() && end_ != cur_) err_ = "truncated BAM record";
                return false;
            }
        }
        const uint32_t bs = rd32(cur_batch_->data.data() + cur_);
        if (bs < 32) { err_ = "corrupt BAM record"; return false; }
        if (end_ - cur_ < (size_t)bs + 4) {
            if (!recs.empty()) break;                             // the rest of this record is in the next batch
            const double tw = now();
            const bool okb = ensure_bytes((size_t)bs + 4);
            t_waited += now() - tw;
            if (!okb) { if (err_.empty()) err_ = "truncated BAM record"; return false; }
        }
        recs.emplace_back(cur_ + 4, bs);
        cur_ += (size_t)bs + 4;
    }
    const double t_indexed = now();
    s_wait_batch += t_waited;
    s_index += t_indexed - t_begin - t_waited;
    // 2. parse in parallel: chunks of consecutive records
    constexpr size_t kChunk = 256;
    const size_t n_chunks = (recs.size() + kChunk - 1) / kChunk;
    chunks.resize(n_chunks);
    const uint8_t *base = cur_batch_->data.data();
    std::atomic<size_t> next{0};
    auto work = [&]() {
        BamRecordView rv;
        std::vector<uint32_t> cg;
        std::vector<size_t> cig_off;
        for (;;) {
            const size_t c = next.fetch_add(1);
            if (c >= n_chunks) break;
            ParsedChunk &pc = chunks[c];
            const size_t a = c * kChunk, b = std::min(recs.size(), a + kChunk);
            pc.n_records = b - a;
            cig_off.clear();
            for (size_t i = a; i < b; ++i) {
                if (!parse_bam_record(base + recs[i].first, recs[i].second, rv, cg, pc.err)) break;
                if (filter.reach && !filter.reach(filter.ctx, rv.tid, rv.pos, rv.end)) continue;
                const BamRecLite l = lite_record(rv, filter.need_hp);
                cig_off.push_back(pc.cigar.size());
                pc.cigar.insert(pc.cigar.end(), l.cigar, l.cigar + l.n_cigar);
                pc.recs.push_back(l);
            }
            for (size_t k = 0; k < pc.recs.size(); ++k)
                pc.recs[k].cigar = pc.recs[k].n_cigar ? pc.cigar.data() + cig_off[k] : nullptr;
        }
    };
    const int nt = (int)std::min<size_t>((size_t)std::max(1, parse_threads), n_chunks);
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    s_parse += now() - t_indexed;
    for (auto &pc : chunks)
        if (!pc.err.empty()) { err_ = pc.err; return false; }
    return true;
}

BamRecLite lite_record(const BamRecordView &rv, bool need_hp)
{
    BamRecLite l{rv.tid, rv.pos, rv.end, 0, nullptr, rv.hp_value, rv.flag, rv.mapq, rv.hp_type, false, false};
    // fails the filter at every locus: never shipped, but kept as a stub without CIGAR so that the caller's counters
    // can tell "unpairable" from "unreachable"
    const bool hp_odd = need_hp && (rv.hp_type == HpType::OtherInt || rv.hp_type == HpType::NotInt);
    if (!hp_odd && (rv.mapq <= 10 || (need_hp && rv.hp_type == HpType::Absent))) return l;
    // is_accidental_2d is only consulted on S ops of reads that passed the filter (call.rs:394): what it would panic on
    // travels as a flag and is raised by the GPU only if the read really pairs with a locus
    bool has_clip = false;
    for (uint32_t k = 0; k < rv.n_cigar && !has_clip; ++k) has_clip = (rv.cigar[k] & 0xF) == 4;
    if (has_clip) l.two_d = is_accidental_2d(rv, &l.sa_panic);
    l.n_cigar = rv.n_cigar;
    l.cigar = rv.cigar;
    return l;
}

bool parse_bam_record(const uint8_t *p, uint32_t block_size, BamRecordView &rec, std::vector<uint32_t> &cg_, std::string &err_)
{
    rec.tid = rdi32(p);
    rec.pos = rdi32(p + 4);
    const uint32_t l_read_name = p[8];
    rec.mapq = p[9];
    uint32_t n_cigar = rd16(p + 12);
    rec.flag = rd16(p + 14);
    const uint32_t l_seq = rd32(p + 16);
    size_t off = 32 + l_read_name;
    const size_t cigar_off = off;
    off += (size_t)n_cigar * 4;
    off += ((size_t)l_seq + 1) / 2 + l_seq;
    if (off > block_size) { err_ = "corrupt BAM record (fields exceed block)"; return false; }

    // aux: HP, SA, CG
    rec.hp_type = HpType::Absent;
    rec.hp_value = 0;
    rec.has_sa = false;
    rec.sa_is_string = false;
    rec.sa.clear();
    const uint8_t *cg_data = nullptr;
    uint32_t cg_count = 0;
    while (off + 3 <= block_size) {
        const uint8_t t0 = p[off], t1 = p[off + 1], ty = p[off + 2];
        off += 3;
        size_t vlen = 0;
        const uint8_t *v = p + off;
        switch (ty) {
        case 'A': case 'c': case 'C': vlen = 1; break;
        case 's': case 'S': vlen = 2; break;
        case 'i': case 'I': case 'f': vlen = 4; break;
        case 'Z': case 'H': {
            const void *z = memchr(v, 0, block_size - off);
            if (!z) { err_ = "corrupt BAM aux string"; return false; }
            vlen = (size_t)((const uint8_t *)z - v) + 1;
            break;
        }
        case 'B': {
            if (off + 5 > block_size) { err_ = "corrupt BAM aux array"; return false; }
            const uint8_t sub = v[0];
            const uint32_t cnt = rd32(v + 1);
            size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
            vlen = 5 + (size_t)cnt * es;
            if (t0 == 'C' && t1 == 'G' && sub == 'I') { cg_data = v + 5; cg_count = cnt; }
            break;
        }
        default: err_ = "unknown BAM aux type"; return false;
        }
        if (off + vlen > block_size) { err_ = "corrupt BAM aux field"; return false; }
        if (t0 == 'H' && t1 == 'P') {
            switch (ty) {
            case 'C': rec.hp_type = HpType::U8; rec.hp_value = v[0]; break;
            case 'i': rec.hp_type = HpType::I32; rec.hp_value = rdi32(v); break;
            case 'c': rec.hp_type = HpType::OtherInt; rec.hp_value = (int8_t)v[0]; break;
            case 's': rec.hp_type = HpType::OtherInt; rec.hp_value = (int16_t)rd16(v); break;
            case 'S': rec.hp_type = HpType::OtherInt; rec.hp_value = rd16(v); break;
            case 'I': rec.hp_type = HpType::OtherInt; rec.hp_value = rd32(v); break;
            default: rec.hp_type = HpType::NotInt; break;
            }
        } else if (t0 == 'S' && t1 == 'A') {
            rec.has_sa = true;
            rec.sa_is_string = (ty == 'Z');
            if (ty == 'Z') rec.sa.assign((const char *)v, vlen - 1);
        }
        off += vlen;
    }

    // CIGAR (aligned copy); long CIGARs live in CG:B,I when the in-record CIGAR is <l_seq>S<rlen>N
    const uint8_t *cg_src = p + cigar_off;
    if (cg_data && n_cigar >= 1) {
        const uint32_t w0 = rd32(p + cigar_off);
        if ((w0 & 0xF) == 4 && (w0 >> 4) == l_seq) { cg_src = cg_data; n_cigar = cg_count; }
    }
    cg_.resize(n_cigar);
    if (n_cigar) memcpy(cg_.data(), cg_src, (size_t)n_cigar * 4);
    rec.cigar = cg_.data();
    rec.n_cigar = n_cigar;

    int64_t rlen = 0;
    if (!(rec.flag & 0x4)) {
        for (uint32_t i = 0; i < n_cigar; ++i) {
            const uint32_t op = cg_[i] & 0xF;
            if ((0x18Du >> op) & 1u) rlen += cg_[i] >> 4;       // M,D,N,=,X
        }
    }
    if (rlen == 0) rlen = 1;
    rec.end = (int32_t)(rec.pos + rlen);
    return true;
}

// ---- BamIndexedReader -----------------------------------------------------------------------------
BamIndexedReader::~BamIndexedReader()
{
    if (fp_) fclose(fp_);
}

bool BamIndexedReader::load_block(uint64_t coffset)
{
    if (fseeko(fp_, (off_t)coffset, SEEK_SET) != 0) { err_ = "seek failed"; return false; }
    uint8_t h[12];
    const size_t n = fread(h, 1, 12, fp_);
    block_.clear();
    block_pos_ = 0;
    block_coff_ = coffset;
    if (n == 0) { at_eof_ = true; return false; }
    if (n != 12 || h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) { err_ = "not a BGZF block (bad gzip header)"; return false; }
    const uint16_t xlen = rd16(h + 10);
    uint8_t extra[65536];
    if (fread(extra, 1, xlen, fp_) != xlen) { err_ = "truncated BGZF extra field"; return false; }
    int bsize = -1;
    for (size_t i = 0; i + 4 <= xlen;) {
        const uint16_t slen = rd16(&extra[i + 2]);
        if (extra[i] == 'B' && extra[i + 1] == 'C' && slen == 2 && i + 6 <= xlen) bsize = rd16(&extra[i + 4]);
        i += 4 + slen;
    }
    if (bsize < 0) { err_ = "BGZF block without BC subfield"; return false; }
    const long remaining = (long)bsize + 1 - 12 - xlen;
    if (remaining < 8) { err_ = "corrupt BGZF block size"; return false; }
    comp_.resize((size_t)remaining);
    if (fread(comp_.data(), 1, (size_t)remaining, fp_) != (size_t)remaining) { err_ = "truncated BGZF block"; return false; }
    const uint32_t crc = rd32(&comp_[remaining - 8]), isize = rd32(&comp_[remaining - 4]);
    block_.resize(isize);
    if (!inflate_block(comp_.data(), (size_t)remaining - 8, block_.data(), isize, crc)) { err_ = "BGZF inflate / CRC failure"; return false; }
    next_coff_ = coffset + (uint64_t)bsize + 1;
    total_out_ += isize;
    at_eof_ = false;
    return true;
}

bool BamIndexedReader::read_bytes(void *dst, size_t n)
{
    uint8_t *d = static_cast<uint8_t *>(dst);
    while (n) {
        if (block_pos_ >= block_.size()) {
            if (!load_block(next_coff_)) return false;
            continue;
        }
        const size_t k = std::min(n, block_.size() - block_pos_);
        memcpy(d, block_.data() + block_pos_, k);
        block_pos_ += k;
        d += k;
        n -= k;
    }
    return true;
}

bool BamIndexedReader::open_bam(const std::string &bam_path)
{
    fp_ = fopen(bam_path.c_str(), "rb");
    if (!fp_) { err_ = "cannot open " + bam_path; return false; }
    // header through the block reader
    if (!load_block(0)) { if (err_.empty()) err_ = "empty BAM"; return false; }
    uint8_t b4[4], magic[4];
    if (!read_bytes(magic, 4) || memcmp(magic, "BAM\1", 4) != 0) { if (err_.empty()) err_ = "not a BAM file (bad magic)"; return false; }
    if (!read_bytes(b4, 4)) { err_ = "truncated BAM header"; return false; }
    header_.text.resize(rd32(b4));
    if (!header_.text.empty() && !read_bytes(&header_.text[0], header_.text.size())) { err_ = "truncated BAM header"; return false; }
    if (!read_bytes(b4, 4)) { err_ = "truncated BAM header"; return false; }
    const uint32_t n_ref = rd32(b4);
    for (uint32_t i = 0; i < n_ref; ++i) {
        if (!read_bytes(b4, 4)) { err_ = "truncated BAM reference list"; return false; }
        std::string name(rd32(b4), '\0');
        if (!name.empty() && !read_bytes(&name[0], name.size())) { err_ = "truncated BAM reference list"; return false; }
        if (!name.empty() && name.back() == '\0') name.pop_back();
        if (!read_bytes(b4, 4)) { err_ = "truncated BAM reference list"; return false; }
        header_.ref_names.push_back(name);
        header_.ref_lens.push_back((int64_t)rd32(b4));
    }
    return true;
}

bool BamIndexedReader::load_index(const std::string &bai_path)
{
    FILE *fi = fopen(bai_path.c_str(), "rb");
    if (!fi) { err_ = "cannot open " + bai_path; return false; }
    std::vector<uint8_t> bai;
    uint8_t buf[1 << 16];
    size_t k;
    while ((k = fread(buf, 1, sizeof(buf), fi)) > 0) bai.insert(bai.end(), buf, buf + k);
    fclose(fi);
    size_t p = 0;
    auto need = [&](size_t n) { return p + n <= bai.size(); };
    if (!need(8) || memcmp(bai.data(), "BAI\1", 4) != 0) { err_ = "not a BAI index"; return false; }
    const uint32_t nr = rd32(&bai[4]);
    p = 8;
    index_.resize(nr);
    for (uint32_t r = 0; r < nr; ++r) {
        if (!need(4)) { err_ = "truncated BAI"; return false; }
        const uint32_t n_bin = rd32(&bai[p]);
        p += 4;
        for (uint32_t b = 0; b < n_bin; ++b) {
            if (!need(8)) { err_ = "truncated BAI"; return false; }
            const uint32_t bin = rd32(&bai[p]), n_chunk = rd32(&bai[p + 4]);
            p += 8;
            if (!need((size_t)n_chunk * 16)) { err_ = "truncated BAI"; return false; }
            std::vector<Chunk> ch(n_chunk);
            for (uint32_t c = 0; c < n_chunk; ++c) {
                ch[c].beg = (uint64_t)rd32(&bai[p]) | ((uint64_t)rd32(&bai[p + 4]) << 32);
                ch[c].end = (uint64_t)rd32(&bai[p + 8]) | ((uint64_t)rd32(&bai[p + 12]) << 32);
                p += 16;
            }
            if (bin != 37450) index_[r].bins.emplace_back(bin, std::move(ch));
            else if (n_chunk >= 2) {                                                // 37450 = metadata pseudo-bin (SAM spec 5.2)
                index_[r].n_mapped = (int64_t)ch[1].beg;
                index_[r].n_unmapped = (int64_t)ch[1].end;
            }
        }
        if (!need(4)) { err_ = "truncated BAI"; return false; }
        const uint32_t n_intv = rd32(&bai[p]);
        p += 4;
        if (!need((size_t)n_intv * 8)) { err_ = "truncated BAI"; return false; }
        index_[r].linear.resize(n_intv);
        for (uint32_t i = 0; i < n_intv; ++i) {
            index_[r].linear[i] = (uint64_t)rd32(&bai[p]) | ((uint64_t)rd32(&bai[p + 4]) << 32);
            p += 8;
        }
    }
    if (need(8)) n_no_coor_ = (uint64_t)rd32(&bai[p]) | ((uint64_t)rd32(&bai[p + 4]) << 32);   // optional trailer
    return true;
}

double BamIndexedReader::window_weight(int tid, int64_t beg, int64_t end) const
{
    if (tid < 0 || tid >= (int)index_.size() || index_[tid].linear.empty()) return 1.0;
    const std::vector<uint64_t> &lin = index_[tid].linear;
    const size_t n = lin.size();
    const size_t a = std::min<size_t>((size_t)(std::max<int64_t>(beg, 0) >> 14), n - 1), b = std::min<size_t>((size_t)(std::max<int64_t>(end, 0) >> 14) + 1, n - 1);
    const uint64_t ca = lin[a] >> 16, cb = lin[b] >> 16;
    return 1.0 + (cb > ca ? (double)(cb - ca) : 0.0);
}

std::vector<std::pair<uint64_t, uint64_t>> BamIndexedReader::chunks_for(int tid, int64_t beg, int64_t end) const
{
    std::vector<std::pair<uint64_t, uint64_t>> out;
    if (tid < 0 || tid >= (int)index_.size()) return out;
    for (const Chunk &c : query_chunks(tid, std::max<int64_t>(beg, 0), end)) out.emplace_back(c.beg, c.end);
    return out;
}

std::vector<BamIndexedReader::Chunk> BamIndexedReader::query_chunks(int tid, int64_t beg, int64_t end) const
{
    const RefIndex &ri = index_[tid];
    if (end <= beg) return {};
    // reg2bins (SAM spec 5.3)
    std::vector<uint32_t> want{0};
    const int64_t e = end - 1;
    for (int64_t k = 1 + (beg >> 26); k <= 1 + (e >> 26); ++k) want.push_back((uint32_t)k);
    for (int64_t k = 9 + (beg >> 23); k <= 9 + (e >> 23); ++k) want.push_back((uint32_t)k);
    for (int64_t k = 73 + (beg >> 20); k <= 73 + (e >> 20); ++k) want.push_back((uint32_t)k);
    for (int64_t k = 585 + (beg >> 17); k <= 585 + (e >> 17); ++k) want.push_back((uint32_t)k);
    for (int64_t k = 4681 + (beg >> 14); k <= 4681 + (e >> 14); ++k) want.push_back((uint32_t)k);
    std::sort(want.begin(), want.end());
    uint64_t min_off = 0;
    if (!ri.linear.empty()) {
        const size_t w = (size_t)(beg >> 14);
        min_off = w < ri.linear.size() ? ri.linear[w] : ri.linear.back();
    }
    std::vector<Chunk> out;
    for (const auto &b : ri.bins) {
        if (!std::binary_search(want.begin(), want.end(), b.first)) continue;
        for (const Chunk &c : b.second)
            if (c.end > min_off) out.push_back(c);
    }
    std::sort(out.begin(), out.end(), [](const Chunk &a, const Chunk &b) { return a.beg < b.beg; });
    std::vector<Chunk> merged;
    for (const Chunk &c : out) {
        if (!merged.empty() && c.beg <= merged.back().end) merged.back().end = std::max(merged.back().end, c.end);
        else merged.push_back(c);
    }
    return merged;
}

int64_t cigar_text_to_rlen(const std::string &cigar)
{
    int64_t rlen = 0, num = 0;
    for (char c : cigar) {
        if (c >= '0' && c <= '9') { num = num * 10 + (c - '0'); continue; }
        if (c == 'M' || c == '=' || c == 'X' || c == 'D' || c == 'N') rlen += num;
        num = 0;
    }
    return rlen;
}

bool is_accidental_2d(const BamRecordView &rec, bool *panic)
{
    *panic = false;
    if (!rec.has_sa) return false;                                   // call.rs:425-427
    if (!rec.sa_is_string) { *panic = true; return false; }          // call.rs:431
    const char strand = rec.is_reverse() ? '-' : '+';                // call.rs:422
    // call.rs:434: split on ';', ignore empty entries
    std::vector<std::string> entries;
    size_t a = 0;
    while (a <= rec.sa.size()) {
        size_t b = rec.sa.find(';', a);
        if (b == std::string::npos) b = rec.sa.size();
        if (b > a) entries.push_back(rec.sa.substr(a, b - a));
        a = b + 1;
    }
    if (entries.size() > 1) return false;                            // call.rs:436-438
    if (entries.empty()) { *panic = true; return false; }            // sa_entries[0] on an empty Vec
    std::vector<std::string> f;
    a = 0;
    const std::string &e = entries[0];
    while (a <= e.size()) {
        size_t b = e.find(',', a);
        if (b == std::string::npos) b = e.size();
        f.push_back(e.substr(a, b - a));
        a = b + 1;
    }
    if (f.size() < 3 || f[2].empty()) { *panic = true; return false; }   // sa_entry[2] / .next().unwrap()
    if (strand == f[2][0]) return false;                             // call.rs:441-443
    if (f.size() < 4) { *panic = true; return false; }               // sa_entry[3] is only touched after the strand test
    char *endp = nullptr;
    const long long sa_start = strtoll(f[1].c_str(), &endp, 10);     // call.rs:450 (1-based POS used as is)
    if (endp == f[1].c_str() || *endp) { *panic = true; return false; }
    const long long sa_end = sa_start + cigar_text_to_rlen(f[3]);    // call.rs:451
    const long long lo = std::max<long long>(rec.pos, sa_start), hi = std::min<long long>(rec.end, sa_end);
    return lo < hi;                                                  // call.rs:454
}

}  // namespace inqhost
