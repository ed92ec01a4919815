// bam_reader.hpp -- sequential BGZF/BAM decoder on zlib (htslib is not available in this image).
// Replaces what rust-htslib does for the reference's `call` path: header @SQ names/lengths
// (call.rs:161-180) and, per record, reference_start / reference_end (bam_endpos), mapq, strand,
// CIGAR (incl. the CG:B,I long-CIGAR convention), HP and SA aux tags (call.rs:297-299,382,422-423,483).
// SEQ/QUAL are skipped, never copied.
#pragma once

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace inqhost {

struct BamHeader {
    std::string text;
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    int tid(const std::string &name) const;   // -1 if absent
};

// how an integer aux value was typed in the file (rust-htslib Aux variants the reference matches on)
enum class HpType : uint8_t { Absent, U8, I32, OtherInt, NotInt };

struct BamRecordView {
    int32_t tid = -1;
    int32_t pos = -1;
    int32_t end = 0;             // bam_endpos: pos + max(1, reference length); pos + 1 if unmapped
    uint8_t mapq = 0;
    uint16_t flag = 0;
    const uint32_t *cigar = nullptr;   // BAM packed words (points into the record or into the CG tag)
    uint32_t n_cigar = 0;
    HpType hp_type = HpType::Absent;
    int64_t hp_value = 0;
    bool has_sa = false;
    bool sa_is_string = false;
    std::string sa;              // SA:Z value when present
    bool is_reverse() const { return (flag & 0x10) != 0; }
};

// What the `call` driver needs of one record, produced by the parallel parse (BamReader::next_parsed)
struct BamRecLite {
    int32_t tid, pos, end;
    uint32_t n_cigar;
    const uint32_t *cigar;        // into the chunk's own storage; null for a stub (n_cigar 0)
    int64_t hp_value;
    uint16_t flag;
    uint8_t mapq;
    HpType hp_type;
    bool two_d, sa_panic;
};
struct ParsedChunk {
    std::vector<BamRecLite> recs; // the records the filter kept, in file order
    std::vector<uint32_t> cigar;
    uint64_t n_records = 0;       // all records of the chunk
    std::string err;
};
// decides in the parse workers which records are worth keeping: reach(ctx, tid, pos, end) says whether any locus
// window can fetch the record (call.rs:285-288); records with mapq <= 10 and, when need_hp, without an HP tag fail the
// filter everywhere (call.rs:297-300,350-352) -- but a reachable record with an HP tag of an unexpected type is kept
// so that the caller can raise the reference's panic (call.rs:487) in file order
struct RecFilter {
    bool (*reach)(const void *ctx, int32_t tid, int32_t pos, int32_t end) = nullptr;
    const void *ctx = nullptr;
    bool need_hp = false;
};

// Streaming reader: BGZF blocks are read in batches and inflated by a small thread pool, records are
// parsed in file order.
class BamReader {
public:
    BamReader() = default;
    ~BamReader();
    BamReader(const BamReader &) = delete;
    BamReader &operator=(const BamReader &) = delete;

    // returns false and sets error() on failure. gpu_device >= 0: a GPU engine (include/inqbgzf.h) inflates runs of
    // blocks next to the zlib workers, which then also check the CRC32 of its output; if no engine can be created the
    // workers simply do everything
    bool open(const std::string &path, int threads, int gpu_device = -1);
    const BamHeader &header() const { return header_; }
    // next alignment record; false at EOF or on error (check error())
    bool next(BamRecordView &rec);
    // the records of the next inflated batch, parsed on `parse_threads` threads in chunks of consecutive records; the
    // chunks come back in file order and stay valid until the next call. false at EOF or on error.
    bool next_parsed(const RecFilter &filter, int parse_threads, std::vector<ParsedChunk> &chunks);
    const std::string &error() const { return err_; }
    uint64_t bytes_inflated() const { return total_out_; }

private:
    // fixed-capacity, page-aligned host buffer (recycled between batches; page-locked once when the GPU engine is used)
    struct HostBuf {
        uint8_t *p = nullptr;
        size_t cap = 0;
        bool registered = false;
        uint8_t *data() const { return p; }
        bool empty() const { return p == nullptr; }
    };
    // A batch of BGZF blocks: read raw by the I/O thread, inflated block by block by the worker pool and / or in
    // runs by the GPU engine, parsed by the caller. `data` starts with kSlack unused bytes so that the unconsumed
    // tail of the previous batch can be moved in front of it without copying the batch.
    struct BlockRef {
        size_t in_off, in_len;                     // raw deflate payload inside `comp`
        size_t out_off, out_len;
        uint32_t crc;
    };
    struct Batch {
        HostBuf data, comp;
        std::vector<BlockRef> blocks;
        size_t size = 0;                           // kSlack + inflated payload bytes
        size_t next_block = 0, done_blocks = 0;    // guarded by mu_
        bool eof = false, bad = false;
        std::string err;
    };
    struct CrcRange { Batch *b; size_t next, end; };   // blocks the GPU inflated: CRC32 still to be checked by a worker
    struct Buffers { HostBuf data, comp; };
    std::vector<Buffers> pool_;                    // recycled buffers (guarded by mu_)
    static constexpr size_t kSlack = 8u << 20;
    static constexpr size_t kInFlight = 6;         // batches read ahead of the parser
    static constexpr int kGpuEngines = 3;          // a run of ~1000 blocks fills a quarter of a B200 (one warp per block, ~10 ms per block):
                                                   // several engines on their own streams keep more blocks in flight
    static constexpr size_t kOutCap = 96u << 20;   // inflated bytes per batch
    static constexpr size_t kMaxBlocks = 2048;
    static HostBuf alloc_buf(size_t cap);
    void free_buf(HostBuf &b);
    bool next_batch();                             // make the next batch current (tail preserved)
    bool ensure_bytes(size_t n);                   // at least n unconsumed bytes are contiguous at cur_
    bool parse_header();
    void producer();                               // I/O thread: reads raw batches ahead of the inflaters
    void inflater();                               // worker: CRC checks of GPU-inflated blocks first, then inflates blocks of the oldest unfinished batch
    void gpu_inflater();                           // GPU engine thread: takes runs of blocks off the oldest batch
    bool read_batch(Batch &b);

    int fd_ = -1;
    int threads_ = 1;
    int gpu_device_ = -1;
    BamHeader header_;
    std::string err_;
    std::unique_ptr<Batch> cur_batch_;
    size_t cur_ = 0, end_ = 0;                     // unconsumed window inside cur_batch_->data
    bool eof_ = false;
    uint64_t total_out_ = 0;
    std::vector<uint32_t> cg_;                     // aligned copy of the record's CIGAR
    const uint8_t *map_ = nullptr;                 // the whole file, memory-mapped read-only
    size_t map_len_ = 0, map_pos_ = 0;             // map_pos_: next block header (I/O thread only)

    std::thread producer_;
    std::vector<std::thread> gpu_threads_;
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_;                   // consumer + producer
    std::condition_variable cv_work_;              // inflaters
    std::deque<std::unique_ptr<Batch>> queue_;     // in file order; the head is handed to the parser once complete
    std::deque<CrcRange> crc_;                     // guarded by mu_
    bool stop_ = false, producer_done_ = false;
    std::atomic<uint64_t> gpu_blocks_{0}, gpu_bytes_{0};
public:
    // blocks / bytes inflated by the GPU engine so far
    uint64_t gpu_blocks() const { return gpu_blocks_.load(); }
    uint64_t gpu_bytes() const { return gpu_bytes_.load(); }
    // seconds the consumer spent waiting for an inflated batch / walking record boundaries / in the parallel parse
    double s_wait_batch = 0, s_index = 0, s_parse = 0;
private:
};

// Parses one BAM alignment record body (the bytes after block_size) in place. `cg` receives an aligned
// copy of the CIGAR (from the record or from the CG:B,I tag). Returns false and sets err on corruption.
bool parse_bam_record(const uint8_t *body, uint32_t block_size, BamRecordView &rec, std::vector<uint32_t> &cg,
                      std::string &err);

// Random access through a .bai index (SAM spec 5.2) for small panels: the records htslib's
// fetch(tid, beg, end) yields -- tid match, pos < end, endpos > beg -- in file order
// (replaces IndexedReader::fetch, call.rs:288,338; SURVEY 8f rank 2).
class BamIndexedReader {
public:
    ~BamIndexedReader();
    bool open_bam(const std::string &bam_path);        // header only
    bool load_index(const std::string &bai_path);
    bool has_index() const { return !index_.empty(); }
    // what the index itself says (no BAM needed): references, the metadata pseudo-bin's mapped / unmapped read
    // counts of a reference (-1 when the pseudo-bin is absent), and the merged chunk list fetch() would read
    size_t n_refs() const { return index_.size(); }
    int64_t n_mapped(int tid) const { return tid >= 0 && tid < (int)index_.size() ? index_[tid].n_mapped : -1; }
    int64_t n_unmapped(int tid) const { return tid >= 0 && tid < (int)index_.size() ? index_[tid].n_unmapped : -1; }
    uint64_t n_no_coor() const { return n_no_coor_; }
    std::vector<std::pair<uint64_t, uint64_t>> chunks_for(int tid, int64_t beg, int64_t end) const;
    // 1 + compressed BAM bytes between the linear-index entries of the 16 kb windows around [beg, end): a cheap
    // proxy of the reads piled up there (used to balance catalog shards)
    double window_weight(int tid, int64_t beg, int64_t end) const;
    const BamHeader &header() const { return header_; }
    const std::string &error() const { return err_; }
    uint64_t bytes_inflated() const { return total_out_; }
    // calls f(rec, virtual_offset_of_record) for every record of the query; false on error
    template <typename F>
    bool fetch(int tid, int64_t beg, int64_t end, F f);

private:
    struct Chunk { uint64_t beg, end; };
    struct RefIndex {
        std::vector<std::pair<uint32_t, std::vector<Chunk>>> bins;
        std::vector<uint64_t> linear;
        int64_t n_mapped = -1, n_unmapped = -1;
    };
    bool load_block(uint64_t coffset);             // inflate the block at file offset coffset
    bool read_bytes(void *dst, size_t n);          // from the current position, across blocks
    std::vector<Chunk> query_chunks(int tid, int64_t beg, int64_t end) const;
    uint64_t tell() const { return (block_coff_ << 16) | (uint64_t)block_pos_; }

    FILE *fp_ = nullptr;
    BamHeader header_;
    std::string err_;
    std::vector<RefIndex> index_;
    uint64_t n_no_coor_ = 0;
    std::vector<uint8_t> block_, rec_, comp_;
    uint64_t block_coff_ = 0, next_coff_ = 0;
    size_t block_pos_ = 0;
    bool at_eof_ = false;
    uint64_t total_out_ = 0;
    std::vector<uint32_t> cg_;
};

template <typename F>
bool BamIndexedReader::fetch(int tid, int64_t beg, int64_t end, F f)
{
    if (tid < 0 || tid >= (int)index_.size()) return true;
    if (beg < 0) beg = 0;
    const std::vector<Chunk> chunks = query_chunks(tid, beg, end);
    BamRecordView rec;
    for (const Chunk &c : chunks) {
        if (!load_block(c.beg >> 16)) return err_.empty();
        block_pos_ = (size_t)(c.beg & 0xFFFF);
        for (;;) {
            // normalise the position to the start of the next block when this one is exhausted
            while (block_pos_ >= block_.size() && !at_eof_) {
                if (!load_block(next_coff_)) break;
            }
            if (at_eof_ && block_pos_ >= block_.size()) break;
            const uint64_t v = tell();
            if (v >= c.end) break;
            uint8_t b4[4];
            if (!read_bytes(b4, 4)) return err_.empty();
            const uint32_t bs = (uint32_t)b4[0] | ((uint32_t)b4[1] << 8) | ((uint32_t)b4[2] << 16) | ((uint32_t)b4[3] << 24);
            if (bs < 32) { err_ = "corrupt BAM record"; return false; }
            rec_.resize(bs);
            if (!read_bytes(rec_.data(), bs)) { if (err_.empty()) err_ = "truncated BAM record"; return false; }
            if (!parse_bam_record(rec_.data(), bs, rec, cg_, err_)) return false;
            if (rec.tid != tid || (int64_t)rec.pos >= end) return true;     // coordinate-sorted: nothing further
            if ((int64_t)rec.end > beg) f(rec, v);
        }
    }
    return err_.empty();
}

// BGZF blocks inflated by the own decoder (inflate_fast.hpp) / by zlib (fallback), process-wide
void inflate_counters(uint64_t *fast, uint64_t *zlib_fallback);
// every BGZF block of a file through both decoders, single-threaded: byte comparison + MB/s of each (JSON in *report)
bool bgzf_selfcheck(const std::string &path, std::string *report);

// call.rs:461-477
int64_t cigar_text_to_rlen(const std::string &cigar);
// call.rs:415-459 ; *panic set when the reference would panic (SA not a string)
bool is_accidental_2d(const BamRecordView &rec, bool *panic);
// What the `call` driver keeps of a record that some locus window reaches. A record with mapq <= 10 or, when need_hp,
// without an HP tag fails the filter at every locus (call.rs:297-300,350-352) and becomes a stub without CIGAR, unless
// its HP tag has a type the reference panics on (call.rs:487). Otherwise the CIGAR points into rv and, for a record
// with a soft clip, two_d / sa_panic are what is_accidental_2d says.
BamRecLite lite_record(const BamRecordView &rv, bool need_hp);

}  // namespace inqhost
