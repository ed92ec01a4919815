// inflate_fast.hpp -- one-shot raw DEFLATE (RFC 1951) decoder for BGZF blocks: the whole compressed block
// and the exact output size are known up front, so there is no streaming state, no window copy and no
// per-byte bounds bookkeeping in the hot loop. Written for the host ingest of `inquistr-b200 call`
// (SURVEY 8f rank 1), where zlib's inflate is the bottleneck: 64-bit bit buffer refilled once per symbol
// group, two-level decode tables (11-bit litlen, 8-bit distance primary tables), word-wise match copies.
// Anything unexpected (invalid code, overrun, size mismatch) returns false and the caller falls back to
// zlib; the caller also verifies the block's CRC32, so a decoder bug can never corrupt the output silently.
#pragma once

#include <cstdint>
#include <cstring>

namespace inqhost {

class FastInflater {
public:
    // decodes exactly out_len bytes from in[0, in_len); in must be readable up to in + in_len + 8
    // (a BGZF payload is followed by its 8-byte CRC32/ISIZE trailer)
    bool inflate(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len);

private:
    enum { kReady = 0, kDone = 1, kFail = 2 };
    static constexpr size_t kFastMargin = 320;
    void start(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len);
    int prepare();
    int fast_single();
    bool finish_block(bool eob);
    // the fast loop may run: room for its unchecked stores, input left for its unconditional loads, a sane bit count
    bool fast_ok() const { return (size_t)(out_end_ - out_) > kFastMargin && in_ <= in_end_ && bitcnt_ >= 0; }
    uint8_t *out_ = nullptr, *out_begin_ = nullptr, *out_end_ = nullptr;
    bool bfinal_ = false, finished_ = false;
    static constexpr int kLitBits = 11, kDistBits = 8;
    static constexpr uint32_t kTypeLiteral = 0, kTypeBase = 1, kTypeEob = 2, kTypeSub = 3;
    // Table entry (0 = invalid), laid out for the fewest instructions in the symbol loop:
    //   bits 0-7   everything the entry takes from the stream at this level: a literal's or the end-of-block code, a
    //              length / distance code PLUS its extra bits (one shift advances the buffer), the primary index bits in
    //              front of a sub-table
    //   bits 8-11  base entries: the code bits alone (the extra bits start there in a copy of the buffer; bits 12-13 are
    //              clear in a base entry, so (e >> 8) is a valid 6-bit shift count as it stands); sub entries: index bits
    //   bit 12 sub-table pointer, bit 13 end of block, bit 14 length / distance base, bit 15 literal
    //   bits 16-31 literal byte | base value | sub-table offset
    static constexpr uint32_t kSubFlag = 1u << 12, kEobFlag = 1u << 13, kBaseFlag = 1u << 14, kLitFlag = 1u << 15;
    static uint32_t make(uint32_t type, uint32_t bits, uint32_t extra, uint32_t value)
    {
        switch (type) {
        case kTypeLiteral: return bits | kLitFlag | (value << 16);
        case kTypeEob: return bits | kEobFlag;
        case kTypeBase: return (bits + extra) | (bits << 8) | kBaseFlag | (value << 16);
        default: return bits | (extra << 8) | kSubFlag | (value << 16);      // sub-table: `extra` = its index bits
        }
    }
    static uint32_t entry_bits(uint32_t e) { return e & 0xFFu; }
    bool build(const uint8_t *lens, int n, int primary_bits, uint32_t *table, int table_cap, bool is_dist);
    bool read_dynamic_header();
    void load_fixed();

    uint32_t lit_[(1 << kLitBits) + 2048];
    uint32_t dist_[(1 << kDistBits) + 1024];
    bool fixed_loaded_ = false;

    // bit reader
    const uint8_t *in_ = nullptr, *in_end_ = nullptr;   // in_end_: end of the payload
    uint64_t bitbuf_ = 0;
    int bitcnt_ = 0;
    const uint8_t *in_begin_ = nullptr;
    // Loads whole bytes until the buffer holds >= 56 bits. The 8 trailer bytes after the payload are readable, so a
    // load may pull in bytes that are not payload; consuming them is detected at the end (consumed_ok). Once the
    // pointer has passed the payload nothing more is loaded: the buffer runs dry into zero bits, bitcnt_ goes negative.
    inline void refill()
    {
        if (in_ <= in_end_ && bitcnt_ >= 0) {
            uint64_t w;
            memcpy(&w, in_, 8);
            bitbuf_ |= w << bitcnt_;
            in_ += (63 - bitcnt_) >> 3;
            bitcnt_ |= 56;
        }
    }
    inline bool consumed_ok() const { return (int64_t)(in_ - in_begin_) * 8 - bitcnt_ <= (int64_t)(in_end_ - in_begin_) * 8; }
    inline uint32_t peek(int n) const { return (uint32_t)(bitbuf_ & ((1ull << n) - 1)); }
    inline void consume(int n) { bitbuf_ >>= n; bitcnt_ -= n; }
};

namespace inflate_detail {
static const uint16_t kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
static const uint8_t kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
static const uint16_t kDistBase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
static const uint8_t kDistExtra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
// kExtraMask[n] = n low bits set (n <= 15); kTotalMask[n] likewise for 64-bit values (n <= 28: code + extra bits)
static const uint32_t kExtraMask[16] = {0x0, 0x1, 0x3, 0x7, 0xF, 0x1F, 0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF, 0x3FFF, 0x7FFF};
static const uint64_t kTotalMask[32] = {0x0, 0x1, 0x3, 0x7, 0xF, 0x1F, 0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF, 0x3FFF, 0x7FFF, 0xFFFF,
                                        0x1FFFF, 0x3FFFF, 0x7FFFF, 0xFFFFF, 0x1FFFFF, 0x3FFFFF, 0x7FFFFF, 0xFFFFFF, 0x1FFFFFF, 0x3FFFFFF, 0x7FFFFFF,
                                        0xFFFFFFF, 0x1FFFFFFF, 0x3FFFFFFF, 0x7FFFFFFF};
static const uint8_t kClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
inline uint32_t bitrev(uint32_t v, int n)              // the low n (<= 16) bits of v, reversed
{
    v = ((v & 0x5555u) << 1) | ((v >> 1) & 0x5555u);
    v = ((v & 0x3333u) << 2) | ((v >> 2) & 0x3333u);
    v = ((v & 0x0F0Fu) << 4) | ((v >> 4) & 0x0F0Fu);
    v = ((v & 0x00FFu) << 8) | ((v >> 8) & 0x00FFu);
    return v >> (16 - n);
}
}  // namespace inflate_detail

// canonical Huffman code lengths -> two-level decode table indexed by the next bits of the (LSB-first) stream
inline bool FastInflater::build(const uint8_t *lens, int n, int P, uint32_t *table, int table_cap, bool is_dist)
{
    using namespace inflate_detail;
    int count[16] = {0};
    for (int i = 0; i < n; ++i) count[lens[i]]++;
    count[0] = 0;
    // over-subscription check; incomplete codes are tolerated (unfilled entries stay invalid)
    int left = 1;
    for (int l = 1; l <= 15; ++l) {
        left <<= 1;
        left -= count[l];
        if (left < 0) return false;
    }
    uint32_t next_code[16];
    uint32_t code = 0;
    for (int l = 1; l <= 15; ++l) {
        code = (code + (uint32_t)count[l - 1]) << 1;
        next_code[l] = code;
    }
    const int psize = 1 << P;
    memset(table, 0, (size_t)psize * sizeof(uint32_t));
    // pass 1 for long codes: deepest code below every primary prefix
    uint8_t sub_bits[1 << kLitBits];
    bool any_long = false;
    for (int l = P + 1; l <= 15; ++l) any_long = any_long || count[l] != 0;
    if (any_long) {
        memset(sub_bits, 0, (size_t)psize);
        uint32_t nc[16];
        memcpy(nc, next_code, sizeof(nc));
        for (int s = 0; s < n; ++s) {
            const int l = lens[s];
            if (l <= P) { if (l) nc[l]++; continue; }
            const uint32_t rev = bitrev(nc[l]++, l);
            const uint32_t prefix = rev & (uint32_t)(psize - 1);
            if (l - P > sub_bits[prefix]) sub_bits[prefix] = (uint8_t)(l - P);
        }
        int off = psize;
        for (int p = 0; p < psize; ++p)
            if (sub_bits[p]) {
                const int sz = 1 << sub_bits[p];
                if (off + sz > table_cap) return false;
                memset(table + off, 0, (size_t)sz * sizeof(uint32_t));
                table[p] = make(kTypeSub, (uint32_t)P, sub_bits[p], (uint32_t)off);
                off += sz;
            }
    }
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        if (!l) continue;
        const uint32_t rev = bitrev(next_code[l]++, l);
        uint32_t type, extra = 0, value;
        if (is_dist) {
            if (s >= 30) continue;                        // distance codes 30/31 never occur in valid data: entries stay invalid
            type = kTypeBase; extra = kDistExtra[s]; value = kDistBase[s];
        } else if (s < 256) {
            type = kTypeLiteral; value = (uint32_t)s;
        } else if (s == 256) {
            type = kTypeEob; value = 0;
        } else {
            if (s > 285) continue;                        // 286/287 take part in the fixed code's construction only
            type = kTypeBase; extra = kLenExtra[s - 257]; value = kLenBase[s - 257];
        }
        if (l <= P) {
            const uint32_t e = make(type, (uint32_t)l, extra, value);
            for (uint32_t i = rev; i < (uint32_t)psize; i += 1u << l) table[i] = e;
        } else {
            const uint32_t prefix = rev & (uint32_t)(psize - 1);
            const uint32_t pe = table[prefix];
            const uint32_t sb = (pe >> 8) & 15u, off = pe >> 16;
            const uint32_t e = make(type, (uint32_t)(l - P), extra, value);
            for (uint32_t i = rev >> P; i < (1u << sb); i += 1u << (l - P)) table[off + i] = e;
        }
    }
    return true;
}

inline void FastInflater::load_fixed()
{
    // RFC 1951 3.2.6; symbols 286/287 and distance codes 30/31 exist only to complete the codes
    uint8_t lens[288];
    for (int i = 0; i < 144; ++i) lens[i] = 8;
    for (int i = 144; i < 256; ++i) lens[i] = 9;
    for (int i = 256; i < 280; ++i) lens[i] = 7;
    for (int i = 280; i < 288; ++i) lens[i] = 8;
    build(lens, 288, kLitBits, lit_, (int)(sizeof(lit_) / sizeof(lit_[0])), false);
    uint8_t dl[32];
    for (int i = 0; i < 32; ++i) dl[i] = 5;
    build(dl, 32, kDistBits, dist_, (int)(sizeof(dist_) / sizeof(dist_[0])), true);
}

inline bool FastInflater::read_dynamic_header()
{
    using namespace inflate_detail;
    refill();
    const int hlit = (int)peek(5) + 257; consume(5);
    const int hdist = (int)peek(5) + 1; consume(5);
    const int hclen = (int)peek(4) + 4; consume(4);
    if (hlit > 286 || hdist > 30) return false;
    uint8_t cl[19] = {0};
    for (int i = 0; i < hclen; ++i) {
        if (bitcnt_ < 3) refill();
        cl[kClOrder[i]] = (uint8_t)peek(3);
        consume(3);
    }
    uint32_t cltab[1 << 7];
    if (!build(cl, 19, 7, cltab, 1 << 7, false)) return false;      // symbols 0..18 decode as "literals"
    uint8_t lens[286 + 30 + 138];
    int i = 0;
    const int total = hlit + hdist;
    while (i < total) {
        if (bitcnt_ < 7 + 7) refill();
        const uint32_t e = cltab[peek(7)];
        if (!(e & kLitFlag)) return false;
        consume((int)(e & 0xFFu));
        const uint32_t sym = e >> 16;
        if (sym < 16) { lens[i++] = (uint8_t)sym; continue; }
        int rep;
        uint8_t v = 0;
        if (sym == 16) {
            if (i == 0) return false;
            v = lens[i - 1];
            rep = 3 + (int)peek(2); consume(2);
        } else if (sym == 17) {
            rep = 3 + (int)peek(3); consume(3);
        } else {
            rep = 11 + (int)peek(7); consume(7);
        }
        if (i + rep > total) return false;
        memset(lens + i, v, (size_t)rep);
        i += rep;
    }
    if (lens[256] == 0) return false;                     // no end-of-block code
    if (!build(lens, hlit, kLitBits, lit_, (int)(sizeof(lit_) / sizeof(lit_[0])), false)) return false;
    if (!build(lens + hlit, hdist, kDistBits, dist_, (int)(sizeof(dist_) / sizeof(dist_[0])), true)) return false;
    fixed_loaded_ = false;
    return true;
}

inline void FastInflater::start(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len)
{
    in_ = in_begin_ = in;
    in_end_ = in + in_len;
    bitbuf_ = 0;
    bitcnt_ = 0;
    out_ = out_begin_ = out;
    out_end_ = out + out_len;
    bfinal_ = false;
    finished_ = false;
}

// block headers (and whole stored blocks) up to the first symbol of a Huffman block
inline int FastInflater::prepare()
{
    for (;;) {
        if (finished_) return kDone;
        refill();
        bfinal_ = peek(1) != 0;
        const uint32_t btype = (uint32_t)(bitbuf_ >> 1) & 3u;
        consume(3);
        if (btype == 0) {
            // stored: skip to the byte boundary, LEN / NLEN, raw bytes
            if (bitcnt_ < 0) return kFail;
            consume(bitcnt_ & 7);
            // unread bytes sit in the bit buffer: step the input pointer back to the first unconsumed byte
            const uint8_t *p = in_ - (bitcnt_ >> 3);
            if (p + 4 > in_end_) return kFail;
            const uint32_t len = (uint32_t)p[0] | ((uint32_t)p[1] << 8), nlen = (uint32_t)p[2] | ((uint32_t)p[3] << 8);
            if ((len ^ 0xFFFFu) != nlen) return kFail;
            p += 4;
            if (p + len > in_end_ || out_ + len > out_end_) return kFail;
            memcpy(out_, p, len);
            out_ += len;
            in_ = p + len;
            bitbuf_ = 0;
            bitcnt_ = 0;
            if (!consumed_ok()) return kFail;
            if (bfinal_) finished_ = true;
            continue;
        }
        if (btype == 1) {
            if (!fixed_loaded_) { load_fixed(); fixed_loaded_ = true; }
            return kReady;
        }
        if (btype == 2) return read_dynamic_header() ? kReady : kFail;
        return kFail;
    }
}

// One symbol step of the fast loop on the stream whose locals carry the prefix P. (Stepping two independent blocks
// alternately in one loop -- two dependent chains for the out-of-order core -- was measured: the same MB/s, so the chain
// lookup -> shift -> lookup is not what bounds it; the data-dependent literal / match branch is.) Far enough from
// the end of the output (a symbol writes at most 258 + 7 bytes, three literals 4) that nothing needs a bounds check,
// and far enough from the end of the input that every refill is an unconditional 8-byte load (the 8 trailer bytes
// behind the payload are readable); the checked loop of finish_block() ends the block. The reader's state lives in
// locals: the byte stores through `out` may alias the members as far as the compiler can tell. P##e is always the
// litlen entry for the bits at the front of the buffer, loaded one step ahead: after a match it is fetched before the
// copy, so the table latency hides behind it. Sets P##ex: 1 end of block, 2 invalid stream.
#define INQ_REFILL(P)                                  \
    do {                                               \
        uint64_t w_;                                   \
        memcpy(&w_, P##in, 8);                         \
        P##bb |= w_ << P##bc;                          \
        P##in += (63 - P##bc) >> 3;                    \
        P##bc |= 56;                                   \
    } while (0)
#define INQ_FAST_STEP(P)                                                                                              \
    do {                                                                                                              \
        uint32_t e = P##e;                                                                                            \
        if (e & kLitFlag) {                                                                                           \
            /* a run of literals: up to four primary-table codes (4 x 11 bits) on one refill. (A table that retires */  \
            /* two or three literals per lookup was measured: slower on both the level-1 and the level-6 streams --  */  \
            /* 1.0 to 1.3 literals per lookup there -- and it costs 10 k cycles per block to build.) */                 \
            P##bb >>= (e & 0xFFu);                                                                                    \
            P##bc -= (int)(e & 0xFFu);                                                                                \
            *P##out++ = (uint8_t)(e >> 16);                                                                           \
            e = P##lit[(uint32_t)P##bb & kLitMask];                                                                   \
            if (e & kLitFlag) {                                                                                       \
                P##bb >>= (e & 0xFFu);                                                                                \
                P##bc -= (int)(e & 0xFFu);                                                                            \
                *P##out++ = (uint8_t)(e >> 16);                                                                       \
                e = P##lit[(uint32_t)P##bb & kLitMask];                                                               \
                if (e & kLitFlag) {                                                                                   \
                    P##bb >>= (e & 0xFFu);                                                                            \
                    P##bc -= (int)(e & 0xFFu);                                                                        \
                    *P##out++ = (uint8_t)(e >> 16);                                                                   \
                    e = P##lit[(uint32_t)P##bb & kLitMask];                                                           \
                    if (e & kLitFlag) {                                                                               \
                        P##bb >>= (e & 0xFFu);                                                                        \
                        P##bc -= (int)(e & 0xFFu);                                                                    \
                        *P##out++ = (uint8_t)(e >> 16);                                                               \
                    }                                                                                                 \
                }                                                                                                     \
            }                                                                                                         \
            INQ_REFILL(P);                                                                                            \
            P##e = P##lit[(uint32_t)P##bb & kLitMask];                                                                \
            break;                                                                                                    \
        }                                                                                                             \
        if (__builtin_expect(!(e & kBaseFlag), 0)) {                                                                  \
            /* rare: a code longer than the primary index, the end of the block, or an invalid entry */               \
            if (e & kSubFlag) {                                                                                       \
                P##bb >>= kLitBits;                                                                                   \
                P##bc -= kLitBits;                                                                                    \
                e = P##lit[(e >> 16) + ((uint32_t)P##bb & kExtraMask[(e >> 8) & 15u])];                               \
                if (e & kLitFlag) {                                                                                   \
                    /* (a long literal code: at most 15 bits gone) */                                                 \
                    P##bb >>= (e & 0xFFu);                                                                            \
                    P##bc -= (int)(e & 0xFFu);                                                                        \
                    *P##out++ = (uint8_t)(e >> 16);                                                                   \
                    INQ_REFILL(P);                                                                                    \
                    P##e = P##lit[(uint32_t)P##bb & kLitMask];                                                        \
                    break;                                                                                            \
                }                                                                                                     \
            }                                                                                                         \
            if (e & kEobFlag) {                                                                                       \
                P##bb >>= (e & 0xFFu);                                                                                \
                P##bc -= (int)(e & 0xFFu);                                                                            \
                P##ex = 1;                                                                                            \
                break;                                                                                                \
            }                                                                                                         \
            if (!(e & kBaseFlag)) { P##ex = 2; break; }                                                               \
        }                                                                                                             \
        /* length: one shift on the chain (code + extra bits); the extra bits are read from the copy: everything  */ \
        /* below the entry's total, shifted down by its code bits ((e >> 8) is a clean 6-bit count in a base entry) */ \
        const uint64_t sl = P##bb;                                                                                    \
        P##bb >>= (e & 0xFFu);                                                                                        \
        P##bc -= (int)(e & 0xFFu);                                                                                    \
        const uint32_t len = (e >> 16) + (uint32_t)((sl & kTotalMask[e & 0xFFu]) >> ((e >> 8) & 63u));                \
        uint32_t d = P##dtab[(uint32_t)P##bb & kDistMask];                                                            \
        if (__builtin_expect(!(d & kBaseFlag), 0)) {                                                                  \
            if (!(d & kSubFlag)) { P##ex = 2; break; }                                                                \
            P##bb >>= kDistBits;                                                                                      \
            P##bc -= kDistBits;                                                                                       \
            d = P##dtab[(d >> 16) + ((uint32_t)P##bb & kExtraMask[(d >> 8) & 15u])];                                  \
            if (!(d & kBaseFlag)) { P##ex = 2; break; }                                                               \
        }                                                                                                             \
        const uint64_t sd = P##bb;                                                                                    \
        P##bb >>= (d & 0xFFu);                                                                                        \
        P##bc -= (int)(d & 0xFFu);                                                                                    \
        const uint32_t dist = (d >> 16) + (uint32_t)((sd & kTotalMask[d & 0xFFu]) >> ((d >> 8) & 63u));               \
        if (dist > (size_t)(P##out - P##out_begin)) { P##ex = 2; break; }                                             \
        /* next symbol's entry first (at most 48 of the 56 bits are gone: the refill cannot be skipped) */            \
        INQ_REFILL(P);                                                                                                \
        P##e = P##lit[(uint32_t)P##bb & kLitMask];                                                                    \
        const uint8_t *src = P##out - dist;                                                                           \
        uint8_t *dst = P##out;                                                                                        \
        P##out += len;                                                                                                \
        if (dist >= 8) {                                                                                              \
            do {                                                                                                      \
                uint64_t w;                                                                                           \
                memcpy(&w, src, 8);                                                                                   \
                memcpy(dst, &w, 8);                                                                                   \
                src += 8;                                                                                             \
                dst += 8;                                                                                             \
            } while (dst < P##out);                                                                                   \
        } else if (dist == 1) {                                                                                       \
            memset(dst, *src, len);                                                                                   \
        } else {                                                                                                      \
            /* short period: plain forward byte copy (source and destination overlap) */                              \
            for (uint32_t k = 0; k < len; ++k) dst[k] = src[k];                                                       \
        }                                                                                                             \
    } while (0)
#define INQ_FAST_LOAD(P, obj)                                                                                          \
    const uint8_t *P##in = (obj).in_;                                                                                 \
    const uint8_t *const P##in_last = (obj).in_end_; /* a load may start here at the latest */                        \
    uint64_t P##bb = (obj).bitbuf_;                                                                                   \
    int P##bc = (obj).bitcnt_;                                                                                        \
    uint8_t *P##out = (obj).out_;                                                                                     \
    uint8_t *const P##out_begin = (obj).out_begin_;                                                                   \
    uint8_t *const P##fast_end = (obj).out_end_ - kFastMargin;                                                        \
    const uint32_t *const P##lit = (obj).lit_, *const P##dtab = (obj).dist_;            \
    int P##ex = 0;                                                                                                    \
    INQ_REFILL(P);                                                                                                    \
    uint32_t P##e = P##lit[(uint32_t)P##bb & kLitMask]
#define INQ_FAST_STORE(P, obj)                                                                                         \
    (obj).in_ = P##in;                                                                                                \
    (obj).bitbuf_ = P##bb;                                                                                            \
    (obj).bitcnt_ = P##bc;                                                                                            \
    (obj).out_ = P##out

// fast loop of one stream; returns 0 (left the fast region), 1 (end of block) or 2 (invalid)
inline int FastInflater::fast_single()
{
    if (!fast_ok()) return 0;
    using inflate_detail::kExtraMask;
    using inflate_detail::kTotalMask;
    constexpr uint32_t kLitMask = (1u << kLitBits) - 1u, kDistMask = (1u << kDistBits) - 1u;
    INQ_FAST_LOAD(a_, *this);
    while (a_out < a_fast_end && a_in <= a_in_last) {
        INQ_FAST_STEP(a_);
        if (a_ex) break;
    }
    INQ_FAST_STORE(a_, *this);
    return a_ex;
}

#undef INQ_FAST_LOAD
#undef INQ_FAST_STORE
#undef INQ_FAST_STEP
#undef INQ_REFILL

// the rest of the current block with every bound checked; `eob`: the fast loop has already consumed the end-of-block code
inline bool FastInflater::finish_block(bool eob)
{
    uint8_t *out = out_;
    while (!eob) {
        refill();                                            // >= 56 bits: enough for one length/distance pair (48)
        uint32_t e = lit_[peek(kLitBits)];
        if (e & kSubFlag) {
            consume(kLitBits);
            e = lit_[(e >> 16) + peek((int)((e >> 8) & 15u))];
        }
        if (!e || (e & kSubFlag)) return false;
        if (e & kLitFlag) {
            consume((int)entry_bits(e));
            if (out >= out_end_) return false;
            *out++ = (uint8_t)(e >> 16);
            continue;
        }
        if (e & kEobFlag) { consume((int)entry_bits(e)); break; }
        const uint32_t cl = (e >> 8) & 15u, xl = entry_bits(e) - cl;
        consume((int)cl);
        const uint32_t len = (e >> 16) + peek((int)xl);
        consume((int)xl);
        uint32_t d = dist_[peek(kDistBits)];
        if (d & kSubFlag) {
            consume(kDistBits);
            d = dist_[(d >> 16) + peek((int)((d >> 8) & 15u))];
        }
        if (!(d & kBaseFlag)) return false;
        const uint32_t cd = (d >> 8) & 15u, xd = entry_bits(d) - cd;
        consume((int)cd);
        const uint32_t dist = (d >> 16) + peek((int)xd);
        consume((int)xd);
        if (dist > (size_t)(out - out_begin_) || len > (size_t)(out_end_ - out)) return false;
        const uint8_t *src = out - dist;
        for (uint32_t k = 0; k < len; ++k) out[k] = src[k];
        out += len;
    }
    out_ = out;
    if (!consumed_ok()) return false;
    if (bfinal_) finished_ = true;
    return true;
}

inline bool FastInflater::inflate(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len)
{
    start(in, in_len, out, out_len);
    for (;;) {
        const int r = prepare();
        if (r == kFail) return false;
        if (r == kDone) break;
        const int ex = fast_single();
        if (ex == 2 || !finish_block(ex == 1)) return false;
    }
    return out_ == out_end_;
}

}  // namespace inqhost
