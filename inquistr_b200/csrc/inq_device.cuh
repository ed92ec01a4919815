// inq_device.cuh -- sm_100a kernels of the `inquiSTR call` hot path.
//
// Reference semantics being reproduced (files under /root/reference/src, v0.13.0):
//   K1  k_join_ranges     read x locus overlap join (ranges)   call.rs:288,338
//   K2  k_cigar_scan      segmented CIGAR scan -> event list   call.rs:377-413 (position cursor + op tests)
//   K2b k_pair_eval       filter, window sum, bucket scatter   call.rs:297-301,349-355,388-403,304,358
//   K3  k_locus_median*   sort / split / support / median      call.rs:308-321,365-369,497-522
//
// Layout in HBM (all structure-of-arrays, see DESIGN.md):
//   reads : contig/ref_start/ref_end int32[R], mapq/hp/flags u8[R], cig_off u64[R+1] (BAM words),
//           unit_off u64[R+1], units u16[U] (the CIGAR stream as 16-bit units, see "CIGAR units" below)
//   loci  : start/end/pmax_end int32[L] sorted by (contig,start), contig_off int64[n_contigs+1]
//   events: uint2{pos1 (1-based anchor, u32), val = (signed len << 1) | is_softclip}[E], ev_off u32[R+1]
//   calls : one segment per locus sized by its candidate count (seg_off u32[L+1]); H1 from the front,
//           H2 from the back (cursor u64[L] = front count | back count << 32); vals u64[#candidates]
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace inq {

// ----------------------------------------------------------------------------------------------
// constants
constexpr int kTileUnits = 16384;           // padding granularity of the device CIGAR stream (32 KB)

constexpr uint32_t kFlagBadHp = 1u << 0;
constexpr uint32_t kFlagMedianEmpty = 1u << 1;
constexpr uint32_t kFlagEventOverflow = 1u << 2;
constexpr uint32_t kFlagValsOverflow = 1u << 3;
constexpr uint32_t kFlagCountOverflow = 1u << 4;
constexpr uint32_t kFlagBadSa = 1u << 5;
constexpr uint32_t kFlagWideCall = 1u << 6;   // a pass with 32-bit call keys met a call outside [-2^29, 2^29)

constexpr uint64_t kDescAggregate = 1ull << 62;
constexpr uint64_t kDescPrefix = 2ull << 62;
constexpr uint64_t kDescValueMask = (1ull << 62) - 1;

constexpr int64_t kCallBias = 1ll << 61;    // keys are (call + bias) << 1 | clip, 63 bits
constexpr uint64_t kKeyHapBit = 1ull << 63;
constexpr uint64_t kKeyInf = ~0ull;

// device-side counters, one struct per ctx
// statistics are accumulated per block into one of kStatSlots copies (a single address would
// serialise hundreds of thousands of atomics in L2); the host adds the copies up
constexpr int kStatSlots = 64;
enum { ST_CANDIDATES = 0, ST_PAIRS, ST_READS_JOINED, ST_WORDS_JOINED, ST_OP_VISITS, ST_COUNT = 8 };

constexpr int kMaxMedianChunks = 48;        // the medians run in catalog chunks so that the result copy of one overlaps the next
struct DevCounters {
    unsigned long long stat[kStatSlots][ST_COUNT];
    unsigned long long n_events;
    unsigned long long ev_alloc;      // event slots handed out to warps (chunks)
    unsigned int flags;
    unsigned int tile_counter;
    unsigned int scan_counter[4];
    unsigned int wt_scan_counter;     // dynamic tile ids of k_exclusive_scan2
    unsigned int big_count[kMaxMedianChunks];  // per chunk of the catalog (see inq_genotype): loci for the CTA path
    unsigned int big_cursor[kMaxMedianChunks];
    unsigned int bad_hp_value;        // diagnostics: HP value and read index of one offending read
    unsigned long long bad_hp_read;
    unsigned long long bad_sa_read;
};

// ----------------------------------------------------------------------------------------------
// small helpers
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t *p)
{
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t *p, uint64_t v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt()
{
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
__device__ __forceinline__ uint32_t lanemask_le()
{
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_le;" : "=r"(m));
    return m;
}

// mbarrier helpers for the TMA tensor loads of k_cigar_scan
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// poll with a short sleep in between so that waiting warps do not burn issue slots
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, uint32_t parity, uint32_t ns)
{
    uint32_t done = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(ns);
    }
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// CIGAR units. BAM words are (len << 4) | op with ops MIDNSHP=X -> 0..8; M,D,N,=,X consume the reference
// (call.rs:384-392,404), I,D,S longer than minlen are events (call.rs:388,394,400). The device keeps the
// stream as 16-bit units written when reads are pushed. A unit carries what the scan asks of an op as bits, so that
// both units of a 32-bit word are tested together with 32-bit arithmetic (k_cigar_scan):
//   bit 15 C: consumes the reference; bits 14-13 sub; bit 12 E: I, D or S; bits 11-0: len
//     M, N, =, X piece   C            len          I   E          len
//     D or long-D head   C | E        len          S   E | sub 1  len
//     payload (below)    sub = 2 payload bits, bits 11-0 = 12 payload bits (C = E = 0: no consumption, no event)
//   - H, P, the invalid codes 9..15 and every op of length 0 are dropped: they consume nothing and are never events;
//   - M, N, = and X longer than 4095 are split into pieces of at most 4095 (consumption adds up);
//   - I, D and S of length >= 4095 are a head with len 4095 followed by two payload units that hold the full
//     length (14 bits each). A long D's head consumes 4095 and is followed by N pieces for the rest, so that
//     consumption still adds up unit by unit.
// So for I/D/S the 12-bit field is the exact length below 4095 and 4095 exactly for a long head: the event test on
// the field is exact for minlen < 4095; a larger minlen looks the heads' full length up (k_cigar_scan<true>).
// The all-zero unit (padding, and a payload of 0) consumes nothing and is never an event.
constexpr uint32_t kUnitLong = 4095;        // field of a long I/D/S head; longest piece of a split op
constexpr uint32_t kUnitLen = 0x0FFFu;
constexpr uint32_t kUnitE = 1u << 12;
constexpr uint32_t kUnitSub = 3u << 13;
constexpr uint32_t kUnitS = 1u << 13;
constexpr uint32_t kUnitC = 1u << 15;

__device__ __forceinline__ bool op_dropped(uint32_t op) { return op > 8u || op == 5u || op == 6u; }
__device__ __forceinline__ bool op_event_class(uint32_t op) { return ((0x16u >> op) & 1u) != 0u; }
// flag bits of the units of a kept op
__device__ __forceinline__ uint32_t op_unit_flags(uint32_t op)
{
    return op == 1u ? kUnitE : op == 2u ? kUnitC | kUnitE : op == 4u ? kUnitE | kUnitS : kUnitC;
}
__device__ __forceinline__ uint32_t split_pieces(uint32_t len) { return (len + kUnitLong - 1u) / kUnitLong; }
__device__ __forceinline__ uint16_t payload_unit(uint32_t p14) { return (uint16_t)(((p14 & 3u) << 13) | (p14 >> 2)); }
__device__ __forceinline__ uint32_t payload_value(uint32_t u) { return ((u & kUnitLen) << 2) | ((u >> 13) & 3u); }
// full length of the long head at unit index h of the stream
__device__ __forceinline__ uint32_t long_head_len(const uint16_t *__restrict__ units, uint64_t h)
{
    return payload_value(__ldg(units + h + 1)) | (payload_value(__ldg(units + h + 2)) << 14);
}

// units that BAM word w becomes
__device__ __forceinline__ uint32_t unit_count(uint32_t w)
{
    const uint32_t op = w & 15u, len = w >> 4;
    if (op_dropped(op) || len == 0u) return 0u;
    if (!op_event_class(op)) return split_pieces(len);
    if (len < kUnitLong) return 1u;
    return op == 2u ? 3u + split_pieces(len - kUnitLong) : 3u;
}
__device__ __forceinline__ void unit_write(uint32_t w, uint16_t *__restrict__ out)
{
    const uint32_t op = w & 15u;
    uint32_t len = w >> 4;
    if (op_dropped(op) || len == 0u) return;
    uint32_t flags = op_unit_flags(op);
    if (op_event_class(op)) {
        if (len < kUnitLong) { out[0] = (uint16_t)(flags | len); return; }
        out[0] = (uint16_t)(flags | kUnitLong);
        out[1] = payload_unit(len & 0x3FFFu);
        out[2] = payload_unit(len >> 14);
        if (op != 2u) return;
        out += 3;
        len -= kUnitLong;
        flags = kUnitC;                     // the rest of a long D: N pieces
    }
    for (; len; len -= min(len, kUnitLong)) *out++ = (uint16_t)(flags | min(len, kUnitLong));
}

template <typename T>
__device__ __forceinline__ T warp_incl_scan(T v)
{
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        T n = __shfl_up_sync(0xffffffffu, v, d);
        if ((int)lane_id() >= d) v += n;
    }
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// first index i in [lo,hi) with a[i] >= key  (a sorted ascending)
__device__ __forceinline__ int lower_bound_i32(const int32_t *__restrict__ a, int lo, int hi, int64_t key)
{
    while (lo < hi) {
        int mid = lo + ((hi - lo) >> 1);
        if ((int64_t)__ldg(a + mid) >= key) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// ----------------------------------------------------------------------------------------------
__global__ void k_rebase_offsets(uint64_t *__restrict__ off, uint64_t n, uint64_t base)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        off[i] += base;
}

// ----------------------------------------------------------------------------------------------
// K1: read x locus overlap join, counting pass. One thread per read, warp-uniform candidate loop,
// warp-aggregated atomics into the per-bucket counters.
//
// unphased (call.rs:297-300): keep iff ref_start <= start_ext && ref_end >= end_ext && mapq > 10
// phased   (call.rs:350-352): keep iff HP present && !(start_ext < ref_start && ref_end < end_ext)
//                             && mapq > 10, among reads fetch() yields (pos < end_ext && endpos > start_ext)
struct ReadView {
    const int32_t *contig, *rs, *re;
    const uint8_t *mapq, *hp, *flags;
    const uint64_t *cig_off;
    uint64_t R;
};
struct LocusView {
    const int64_t *contig_off;
    const int32_t *start, *end, *pmax;
    int n_contigs;
};

__device__ __forceinline__ bool pair_passes(bool unphased, int32_t rs, int32_t re, int32_t lstart, int32_t lend)
{
    // windows as the reference computes them (call.rs:285-286), compared after `as u32` casts
    const uint32_t start_ext = (uint32_t)lstart - 10u, end_ext = (uint32_t)lend + 10u;
    const uint32_t urs = (uint32_t)rs, ure = (uint32_t)re;
    if (unphased) return !(start_ext < urs || ure < end_ext);
    const bool fetched = ((int64_t)rs < (int64_t)end_ext) && ((int64_t)re > (int64_t)start_ext);
    return fetched && !(start_ext < urs && ure < end_ext);
}

__device__ __forceinline__ void candidate_range(bool unphased, const LocusView &lv, int c, int32_t rs, int32_t re,
                                                int &lo, int &hi)
{
    const int l0 = (int)lv.contig_off[c], l1 = (int)lv.contig_off[c + 1];
    if (unphased) {
        lo = lower_bound_i32(lv.start, l0, l1, (int64_t)rs + 10);          // start - 10 >= rs
        hi = lower_bound_i32(lv.start, lo, l1, (int64_t)re - 10 + 1);      // start + 10 <= re (necessary)
    } else {
        hi = lower_bound_i32(lv.start, l0, l1, (int64_t)re + 10);          // start - 10 < re
        lo = lower_bound_i32(lv.pmax, l0, hi, (int64_t)rs - 10 + 1);       // max(end) + 10 > rs
    }
    if (hi < lo) hi = lo;
}

// ---- the same two lower bounds, found by the warp together (k_join_ranges runs under the HBM-saturating CIGAR scan,
// where a dependent L2 round trip costs ~1 us: 2 x 17 of them per read are what the kernel's time is made of).
// Reads arrive coordinate-sorted, so the 32 answers of a warp lie within a few catalog entries of each other:
//   1. one 33-ary search by all lanes for the smallest key of the warp (4-5 round trips instead of 17),
//   2. the 32 entries from there on are loaded once, one per lane, and every lane finds its own bound among them
//      with shuffles (no memory),
//   3. the second bound lies within a 32-entry window of the first one; same trick.
// A lane whose answer falls outside a window (unsorted reads, very long reads) finishes with the plain binary search
// over the rest, and a warp that straddles contigs takes the scalar path: the results are the unique lower bounds
// either way.
__device__ __forceinline__ int warp_lower_bound(const int32_t *__restrict__ a, int lo, int hi, int64_t key)
{
    const int lane = (int)lane_id();
    while (hi - lo > 32) {
        const int n = hi - lo;
        const int p = lo + (int)(((int64_t)(lane + 1) * n) / 33);            // lo < p < hi, increasing with the lane
        const uint32_t m = __ballot_sync(0xffffffffu, (int64_t)__ldg(a + p) >= key);
        const int f = m ? __ffs(m) - 1 : 32;                                 // first probe that is >= key
        const int new_hi = f < 32 ? lo + (int)(((int64_t)(f + 1) * n) / 33) : hi;
        const int new_lo = f > 0 ? lo + (int)(((int64_t)f * n) / 33) + 1 : lo;
        lo = new_lo;
        hi = new_hi;
    }
    const int p = lo + lane;
    const uint32_t m = __ballot_sync(0xffffffffu, p < hi && (int64_t)__ldg(a + p) >= key);
    return m ? lo + __ffs(m) - 1 : hi;
}

// number of entries of the window a[win, win + wn) (wn <= 32, entry j held by lane j in `v`) that are < key
__device__ __forceinline__ int window_count_less(int32_t v, int wn, int64_t key)
{
    int cnt = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int32_t probe = __shfl_sync(0xffffffffu, v, (cnt + step - 1) & 31);
        if (cnt + step - 1 < wn && (int64_t)probe < key) cnt += step;
    }
    const int32_t last = __shfl_sync(0xffffffffu, v, 31);
    if (cnt == 31 && wn == 32 && (int64_t)last < key) cnt = 32;
    return cnt;
}

// all 32 lanes call this; `act` lanes carry a read on contig c (warp-uniform among the active lanes)
__device__ __forceinline__ void candidate_range_warp(bool unphased, const LocusView &lv, int c, bool act, int32_t rs, int32_t re,
                                                     int &lo, int &hi)
{
    const int lane = (int)lane_id();
    const int l0 = (int)lv.contig_off[c], l1 = (int)lv.contig_off[c + 1];
    // first bound: over start[l0, l1)
    const int64_t key1 = unphased ? (int64_t)rs + 10 : (int64_t)re + 10;
    const int64_t big = 0x7fffffffffffffffll;
    int64_t kmin = act ? key1 : big;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) { const int64_t o = __shfl_xor_sync(0xffffffffu, kmin, d); kmin = o < kmin ? o : kmin; }
    const int p1 = warp_lower_bound(lv.start, l0, l1, kmin);
    const int wn1 = min(32, l1 - p1);
    const int32_t v1 = lane < wn1 ? __ldg(lv.start + p1 + lane) : 0;
    const int c1 = window_count_less(v1, wn1, key1);
    int b1 = p1 + c1;
    if (act && c1 == 32 && p1 + 32 < l1) b1 = lower_bound_i32(lv.start, p1 + 32, l1, key1);
    if (unphased) {
        lo = b1;                                                             // start - 10 >= rs
        // hi = lower_bound(start[lo, l1), re - 9): at or after the warp's smallest lo
        const int64_t key2 = (int64_t)re - 10 + 1;
        const int w2 = __reduce_min_sync(0xffffffffu, act ? lo : 0x7fffffff);
        const bool any = w2 != 0x7fffffff;
        const int wn2 = any ? min(32, l1 - w2) : 0;
        const int32_t v2 = lane < wn2 ? __ldg(lv.start + w2 + lane) : 0;
        const int c2 = window_count_less(v2, wn2, key2);
        int b2 = w2 + c2;
        if (act && c2 == 32 && w2 + 32 < l1) b2 = lower_bound_i32(lv.start, w2 + 32, l1, key2);
        hi = b2 > lo ? b2 : lo;
    } else {
        hi = b1;                                                             // start - 10 < re
        // lo = lower_bound(pmax[l0, hi), rs - 9): at most the warp's largest hi, usually within 32 entries below it
        const int64_t key2 = (int64_t)rs - 10 + 1;
        const int hmax = __reduce_max_sync(0xffffffffu, act ? hi : -1);
        const int w2 = hmax - 32 > l0 ? hmax - 32 : l0;
        const int wn2 = hmax > w2 ? min(32, hmax - w2) : 0;
        const int32_t v2 = lane < wn2 ? __ldg(lv.pmax + w2 + lane) : 0;
        const int c2 = window_count_less(v2, wn2, key2);
        int b2 = w2 + c2;
        if (act && c2 == 0 && w2 > l0) b2 = lower_bound_i32(lv.pmax, l0, w2, key2);
        lo = b2 < hi ? b2 : hi;
    }
    if (hi < lo) hi = lo;
}

// K1: per read, the contiguous range [lo, lo+n) of catalog loci whose window it can pair with
// (two lower bounds over the sorted, L2-resident catalog). Instead of visiting the candidates,
// the kernel adds +1/-1 to a difference array; its prefix sum is the number of candidate reads of
// every locus, which sizes that locus' segment of the call buffer (an upper bound on its pairs).
__global__ void __launch_bounds__(256)
k_join_ranges(ReadView rv, LocusView lv, int unphased, uint32_t *__restrict__ cand_lo, uint32_t *__restrict__ cand_n,
              uint32_t *__restrict__ delta /* L+1, zeroed */, DevCounters *__restrict__ ctr)
{
    const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    int lo = 0, n = 0;
    int c = -1;
    int32_t rs = 0, re = 0;
    bool act = false;
    if (r < rv.R) {
        c = rv.contig[r];
        const uint32_t mq = rv.mapq[r], h = rv.hp[r];
        rs = rv.rs[r];
        re = rv.re[r];
        act = c >= 0 && c < lv.n_contigs && mq > 10u && (unphased || h != 0xFFu);
    }
    // one contig for the whole warp? (all warps but the few that straddle a contig boundary)
    const int cmin = __reduce_min_sync(0xffffffffu, act ? c : 0x7fffffff), cmax = __reduce_max_sync(0xffffffffu, act ? c : -1);
    int hi = 0;
    if (cmin == cmax) {
        candidate_range_warp(unphased != 0, lv, cmin, act, rs, re, lo, hi);
    } else if (act) {
        candidate_range(unphased != 0, lv, c, rs, re, lo, hi);
    }
    if (r < rv.R) {
        if (act) n = hi - lo;
        else lo = 0;
        cand_lo[r] = (uint32_t)lo;
        cand_n[r] = (uint32_t)n;
    }
    // +1 at lo, -1 at hi: neighbouring reads share their bounds, so the lanes that hit the same entry send one atomic
    // (11.6 M same-address-heavy atomics per pass were what kept this kernel busy for the whole CIGAR scan)
    {
        const bool has = n > 0;
        const uint32_t mlo = __match_any_sync(0xffffffffu, has ? (uint32_t)lo : 0xFFFFFFFFu);
        const uint32_t mhi = __match_any_sync(0xffffffffu, has ? (uint32_t)hi : 0xFFFFFFFFu);
        if (has) {
            const uint32_t lane = lane_id();
            if ((uint32_t)__ffs(mlo) - 1u == lane) atomicAdd(delta + lo, (uint32_t)__popc(mlo));
            if ((uint32_t)__ffs(mhi) - 1u == lane) atomicAdd(delta + hi, 0u - (uint32_t)__popc(mhi));   // -count (mod 2^32)
        }
    }
    const uint32_t cand_w = __reduce_add_sync(0xffffffffu, (uint32_t)n);
    if (lane_id() == 0 && cand_w)
        atomicAdd(&ctr->stat[(blockIdx.x * 8u + (threadIdx.x >> 5)) % kStatSlots][ST_CANDIDATES], (unsigned long long)cand_w);
}

// ----------------------------------------------------------------------------------------------
// decoupled look-back over tile descriptors (status in the top 2 bits, 62-bit value).
// `stop_at_prefix`: walk back until a tile in kDescPrefix state is found, summing values on the way.
// Called by one full warp. Returns the exclusive carry for tile t.
__device__ __forceinline__ uint64_t lookback(const uint64_t *__restrict__ desc, int64_t t)
{
    uint64_t acc = 0;
    int64_t base = t - 1;
    while (true) {
        const int64_t idx = base - (int64_t)lane_id();
        uint64_t d = kDescPrefix;                       // tiles before 0: prefix 0
        if (idx >= 0) {
            do { d = ld_relaxed_u64(desc + idx); } while ((d >> 62) == 0);
        }
        const uint32_t is_prefix = __ballot_sync(0xffffffffu, (d >> 62) == 2);
        const int first = is_prefix ? (__ffs(is_prefix) - 1) : 32;
        const uint64_t contrib = ((int)lane_id() <= first) ? (d & kDescValueMask) : 0ull;
        acc += warp_sum(contrib);
        if (first < 32) break;
        base -= 32;
    }
    return acc;
}

// ----------------------------------------------------------------------------------------------
// K2: CIGAR scan. Persistent warps stream 4 KB "warp tiles" (2048 units) of the flat CIGAR unit stream
// through per-warp 2-stage shared-memory rings filled by TMA (2-D tensor map, 128B swizzle); each lane
// owns 64 consecutive units (32 words of two units). One pass over the units gives the lane's reference
// consumption (call.rs:384-392,404) and its event masks (I/D/S ops longer than minlen, call.rs:388,394,400);
// two warp scans turn that into warp-local prefixes. Nothing in this kernel depends on another CTA or warp:
// it writes
//   rd_pre : warp-tile-local exclusive prefixes {consumption, events} at the first unit of every read
//            that starts inside the tile (tile_first, built when reads are pushed, names those reads)
//   wt     : totals per warp tile (prefix-summed afterwards by k_exclusive_scan2)
//   evraw  : {bases consumed inside the warp tile before the op, (signed len << 1) | is_S}
//            for every event, stored per warp tile in chunks handed out by one atomic
// and k_read_fixup turns these into per-read event lists with absolute anchors.
// Each unit is read from HBM exactly once (the payload of a long I/D/S head once more, from L2).
struct ScanParams {
    const uint32_t *tile_first;   // [n_wt + 1] first read (index into unit_off, sentinel R included) starting in warp tile t or later
    const uint64_t *unit_off;     // [R + 1] first unit of every read (+ sentinel)
    const uint16_t *units;        // the unit stream (payloads of long heads)
    uint2 *rd_pre;                // [R + 1] {consumption, events} inside the read's warp tile before its first unit
    uint2 *wt;                    // [n_wt] {consumption, events} totals per warp tile (prefix-summed by k_exclusive_scan2 into a second array)
    uint32_t *wt_sbase;           // [n_wt] storage slot of the warp tile's first event
    uint2 *evraw;
    DevCounters *ctr;
    uint64_t raw_cap;             // capacity of evraw (slots)
    uint64_t n_wt;
    uint32_t ev_thr;              // scan_ev_thr(minlen), in both halves
    uint32_t minlen;              // full minlen (the long-head variant)
};

constexpr int kLaneWords = 32;                          // consecutive 32-bit words (unit pairs) per lane
constexpr int kWarpTileUnits = 64 * kLaneWords;         // 2048 units = 4 KB = one TMA box
constexpr int kScanWarps = 24;                          // warps per CTA, each fully autonomous
constexpr int kCtaThreads = kScanWarps * 32;
constexpr int kWarpStages = 2;                          // per-warp ring of TMA boxes
constexpr int kScanMinCtas = 1;
constexpr uint32_t kEvChunk = 1024;                     // event slots a warp takes per atomic
// 0xFFFF in each half of word x whose unit has C set, 0 otherwise: prmt's sign-replicate mode copies bit 15 into
// bytes 0-1 and bit 31 into bytes 2-3 (__byte_perm drops the mode bit of the selector, hence the inline PTX)
__device__ __forceinline__ uint32_t consume_mask(uint32_t x)
{
    uint32_t m;
    asm("prmt.b32 %0, %1, 0, 0xBB99;" : "=r"(m) : "r"(x));
    return m;
}
// consumption of both units of word x as two 16-bit sums (each at most 4095)
__device__ __forceinline__ uint32_t word_consume2(uint32_t x) { return x & consume_mask(x) & 0x0FFF0FFFu; }
__device__ __forceinline__ uint32_t word_consume(uint32_t x)
{
    const uint32_t a = word_consume2(x);
    return (a & 0xFFFFu) + (a >> 16);
}
__device__ __forceinline__ uint32_t unit_consume(uint32_t u) { return (u & kUnitC) ? u & kUnitLen : 0u; }
// Event test on both units of a word: bit 15 / bit 31 of ((x & 0x1FFF1FFF) | 0x80008000) - ev_thr is set exactly when
// that unit has E set and len > minlen. Each half of ev_thr is 0x1000 + minlen + 1 (minlen < 4095), at most 0x1FFF:
// the low half's minuend is >= 0x8000 > ev_thr, so it never borrows from the high half. From minlen 4094 on it is
// 0x1FFF, which selects exactly the long heads (len 4095).
inline uint32_t scan_ev_thr(uint32_t minlen)
{
    return (0x1000u + (minlen < kUnitLong - 1u ? minlen : kUnitLong - 1u) + 1u) * 0x00010001u;
}
__device__ __forceinline__ uint32_t word_events(uint32_t x, uint32_t ev_thr)
{
    return (((x & 0x1FFF1FFFu) | 0x80008000u) - ev_thr) & 0x80008000u;
}

struct ScanSmem {
    alignas(1024) uint32_t stage[kScanWarps][kWarpStages][kWarpTileUnits / 2];   // 128B-swizzled by the TMA tensor map
    uint32_t snap[kScanWarps][kLaneWords / 4][32];                                // per-quad cursor snapshots of every lane
    uint16_t qlist[kScanWarps][32];                                               // unit positions of one round of events
    alignas(8) uint64_t full[kScanWarps][kWarpStages];                            // TMA landed (tx bytes)
};
constexpr size_t kScanSmemBytes = sizeof(ScanSmem) + 1024;   // slack to align the swizzled stages to 1 KB

// `policy`: L2 cache policy of the load. The stream is read exactly once, so its lines are marked evict-first:
// otherwise 5 GB of them flush the catalog and the per-read arrays out of the 126 MB L2, and every probe of the join
// chain that runs next to the scan (and of the pair kernel after it) goes to the saturated HBM instead.
__device__ __forceinline__ void tma_load_tile(void *dst_smem, const CUtensorMap *tmap, uint32_t row, uint64_t *bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(smem_u32(dst_smem)), "l"(tmap), "r"(0), "r"(row), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// A lane's event masks: evA for words 0-15, evB for words 16-31; bit i <-> the low unit of word i (of the 16),
// bit 16 + i <-> its high unit. evs = evA | evB << 32.
// events among the low units of the first nlo words and the high units of the first nhi words of one mask
__device__ __forceinline__ uint32_t events_in_half(uint32_t m, uint32_t nlo, uint32_t nhi)
{
    return __popc(m & (((1u << nlo) - 1u) | (((1u << nhi) - 1u) << 16)));
}
// events among the first k units of a lane: the low units of words [0, (k+1)/2), the high units of words [0, k/2)
__device__ __forceinline__ uint32_t events_before(uint64_t evs, uint32_t k)
{
    const uint32_t nlo = (k + 1u) >> 1, nhi = k >> 1, h = kLaneWords / 2;
    return events_in_half((uint32_t)evs, min(nlo, h), min(nhi, h)) +
           events_in_half((uint32_t)(evs >> 32), nlo - min(nlo, h), nhi - min(nhi, h));
}
// unit index inside the lane of the first event of evs (nonzero) in unit order, and that event's bit
__device__ __forceinline__ uint32_t first_event(uint64_t evs, uint32_t &bit)
{
    const uint32_t b = __ffsll((evs | (evs >> 16)) & 0x0000FFFF0000FFFFull) - 1u;    // lowest word with an event
    bit = (evs >> b) & 1u ? b : b + 16u;                                             // its low unit first
    return 2u * ((b & 15u) | ((b >> 1) & 16u)) + ((bit >> 4) & 1u);
}

// Every warp is an independent pipeline: it owns warp tiles gwid, gwid + W, gwid + 2W, ... (W = warps
// in the grid), a kWarpStages-deep ring of 4 KB shared-memory boxes (one warp tile each) that it fills itself with TMA, and the
// mbarriers of that ring. There is no block-level synchronisation and no producer warp.
// kLongOnly: minlen >= 4095, only long heads can be events and their full length decides.
template <bool kLongOnly>
__global__ void __launch_bounds__(kCtaThreads, kScanMinCtas)
k_cigar_scan(const __grid_constant__ CUtensorMap tmap, ScanParams p)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // keep the pointer in the shared address space (LDS/STS, not generic loads)
    ScanSmem &sm = *reinterpret_cast<ScanSmem *>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr uint32_t kBoxBytes = kWarpTileUnits * 2;
    constexpr uint32_t kRowsPerBox = kWarpTileUnits / 64;       // 128-byte rows
    constexpr uint32_t kLaneUnits = 2 * kLaneWords;
    const uint64_t gwid = (uint64_t)blockIdx.x * kScanWarps + warp, stride = (uint64_t)gridDim.x * kScanWarps;
    uint64_t *full = sm.full[warp];
    const uint64_t l2_policy = l2_evict_first_policy();

    if (lane == 0) {
        for (int s = 0; s < kWarpStages; ++s) mbar_init(&full[s], 1);
        fence_mbar_init();
        for (int s = 0; s < kWarpStages; ++s) {
            const uint64_t gw = gwid + (uint64_t)s * stride;
            if (gw < p.n_wt) {
                mbar_expect_tx(&full[s], kBoxBytes);
                tma_load_tile(sm.stage[warp][s], &tmap, (uint32_t)gw * kRowsPerBox, &full[s], l2_policy);
            }
        }
    }
    __syncwarp();

    const uint32_t ev_thr = p.ev_thr;
    // this lane's kLaneWords consecutive words: quads q0..q0+kLaneWords/4-1 of the box; quad q lives in
    // 128-byte row q/8 at chunk (q%8) ^ (row%8) (128B swizzle) -> conflict-free LDS.128 across the warp
    constexpr uint32_t kQuads = kLaneWords / 4;
    const uint32_t q0 = lane * kQuads;
    uint64_t chunk_cur = 0, chunk_end = 0;                      // this warp's private range of event slots
    // reads that start inside the current warp tile: [tf_lo, tf_hi), lane i holds the first unit of read
    // tf_lo + i. Both are fetched one iteration ahead so that their latency never shows.
    uint32_t tf_lo = 0, tf_hi = 0;
    uint64_t g_cur = 0;
    if (gwid < p.n_wt) {
        tf_lo = __ldg(p.tile_first + gwid);
        tf_hi = __ldg(p.tile_first + gwid + 1);
        if (tf_lo + lane < tf_hi) g_cur = __ldg(p.unit_off + tf_lo + lane);
    }

    for (uint32_t it = 0;; ++it) {
        const uint64_t gw = gwid + (uint64_t)it * stride;       // global warp-tile index
        if (gw >= p.n_wt) break;
        const uint32_t s = it % kWarpStages;
        uint32_t nf_lo = 0, nf_hi = 0;
        if (gw + stride < p.n_wt) {
            nf_lo = __ldg(p.tile_first + gw + stride);
            nf_hi = __ldg(p.tile_first + gw + stride + 1);
        }
        mbar_wait_backoff(&full[s], (it / kWarpStages) & 1u, 32u);
        const uint32_t *stage = sm.stage[warp][s];
        const uint4 *st4 = reinterpret_cast<const uint4 *>(stage);

        // ---- one pass over the lane's words, both units of a word at once. evs: the lane's event masks (see
        //      events_before); snap[j]: bases consumed inside the lane's units before quad j (parked in shared memory below)
        uint32_t c = 0, evA = 0, evB = 0;
        uint32_t snap[kQuads];
#pragma unroll
        for (int j = 0; j < (int)kQuads; ++j) {
            const uint32_t q = q0 + (uint32_t)j, row = q >> 3;
            const uint4 v = st4[row * 8 + ((q & 7u) ^ (row & 7u))];
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
            snap[j] = c;
            uint32_t a = 0;                                       // two 16-bit sums of at most 4 x 4095
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t x = w4[k];
                a += word_consume2(x);
                // after 16 words the event bits of word i sit at bits i and 16 + i. The shifted mask has bits 15 and
                // 31 clear, so an add does the or and fuses with the shift (one LEA.HI)
                uint32_t &ev = j < (int)kQuads / 2 ? evA : evB;
                ev = (ev >> 1) + word_events(x, ev_thr);
            }
            c += (a & 0xFFFFu) + (a >> 16);
        }
        uint64_t evs = evA | ((uint64_t)evB << 32);
        if (kLongOnly) {
            // the candidates are the long heads (field 4095); an event only if the full length is > minlen
            const uint64_t lane_u0 = gw * kWarpTileUnits + lane * kLaneUnits;
            for (uint64_t m = evs; m;) {
                uint32_t bit;
                const uint32_t u = first_event(m, bit);
                m ^= 1ull << bit;
                if (long_head_len(p.units, lane_u0 + u) <= p.minlen) evs ^= 1ull << bit;
            }
        }
        const uint32_t ne = __popcll(evs);
        const uint32_t incl_c = warp_incl_scan(c), incl_e = warp_incl_scan(ne);
        const uint32_t excl_c = incl_c - c, excl_e = incl_e - ne;
        const uint32_t tot_e = __shfl_sync(0xffffffffu, incl_e, 31);
        uint64_t g_nxt = 0;
        if (nf_lo + lane < nf_hi) g_nxt = __ldg(p.unit_off + nf_lo + lane);

        // ---- event slots: contiguous per warp tile, taken from a warp-private chunk
        uint64_t sbase = chunk_cur;
        if (tot_e) {
            if (chunk_end - chunk_cur < tot_e) {
                unsigned long long base = 0;
                const uint32_t n = max(kEvChunk, tot_e);
                if (lane == 0) {
                    base = atomicAdd(&p.ctr->ev_alloc, (unsigned long long)n);
                    // wt_sbase holds 32-bit slots: more than 2^32 slots handed out (stranded chunk remainders included) is an error
                    if (base + n > 0xFFFFFFFFull) atomicOr(&p.ctr->flags, kFlagCountOverflow);
                }
                chunk_cur = __shfl_sync(0xffffffffu, base, 0);
                chunk_end = chunk_cur + n;
                sbase = chunk_cur;
            }
            chunk_cur += tot_e;
        }
        if (lane == 31) {
            p.wt[gw] = make_uint2(incl_c, incl_e);
            p.wt_sbase[gw] = (uint32_t)sbase;
        }

        // ---- position queries. Two things need the tile-local prefix at a unit position: every event
        //      (about 1 % of the units -> {bases consumed before the op, value}) and the first unit of every
        //      read that starts in the tile (-> rd_pre). They are dealt to the lanes 32 at a time (one round
        //      for a typical tile): the lane that owns the unit supplies its scan values by shuffle and its
        //      per-quad snapshot through shared memory; at most 4 words are re-read from the stage.
#pragma unroll
        for (int j = 0; j < (int)kQuads; ++j) sm.snap[warp][j][lane] = snap[j];
        const uint32_t n_starts = tf_hi - tf_lo;
        const uint32_t n_q = tot_e + n_starts;                  // queries [0, tot_e) are the events in unit order
        const uint32_t off_cur = (uint32_t)(g_cur - gw * kWarpTileUnits);    // lane i: first unit of read tf_lo + i
        uint64_t left = evs;
        uint32_t ev_idx = excl_e;
        for (uint32_t base = 0; base < n_q; base += 32) {
            // owners list their events with index in [base, base + 32) in unit order
            while (left && ev_idx < base + 32u) {
                uint32_t bit;
                const uint32_t u = first_event(left, bit);
                left ^= 1ull << bit;
                sm.qlist[warp][ev_idx - base] = (uint16_t)(lane * kLaneUnits + u);
                ++ev_idx;
            }
            __syncwarp();
            const uint32_t qi = base + lane;
            const bool is_ev = qi < tot_e, act = qi < n_q;
            const uint32_t si = qi - tot_e;                     // index of the read start (when !is_ev)
            const uint32_t spos = __shfl_sync(0xffffffffu, off_cur, si & 31u);
            uint32_t pos = 0;
            if (is_ev) pos = sm.qlist[warp][lane];
            else if (act) pos = (si < 32u) ? spos : (uint32_t)(__ldg(p.unit_off + tf_lo + si) - gw * kWarpTileUnits);
            const uint32_t owner = pos / kLaneUnits, k = pos % kLaneUnits;
            const uint32_t xc = __shfl_sync(0xffffffffu, excl_c, owner), xe = __shfl_sync(0xffffffffu, excl_e, owner);
            const uint64_t er = __shfl_sync(0xffffffffu, evs, owner);
            if (act) {
                const uint32_t i = k >> 1, h = k & 1u, j = i >> 2, kk = i & 3u, q = owner * kQuads + j, row = q >> 3;
                const uint4 v = st4[row * 8 + ((q & 7u) ^ (row & 7u))];
                const uint32_t x = kk == 0u ? v.x : kk == 1u ? v.y : kk == 2u ? v.z : v.w;
                // a zero word (two zero units) consumes nothing: blank the words at and after the position
                const uint32_t c_in = xc + sm.snap[warp][j][owner] + word_consume(kk > 0u ? v.x : 0u) +
                                      word_consume(kk > 1u ? v.y : 0u) + word_consume(kk > 2u ? v.z : 0u) +
                                      (h ? unit_consume(x & 0xFFFFu) : 0u);
                if (is_ev) {
                    // E is set: D = C, S = sub 1, I otherwise
                    const uint32_t u = h ? x >> 16 : x & 0xFFFFu;
                    uint32_t len = u & kUnitLen;
                    if (len == kUnitLong) len = long_head_len(p.units, gw * kWarpTileUnits + pos);
                    const int32_t val = (int32_t)(((u & kUnitC) ? (0u - len) : len) << 1) | (int32_t)((u & kUnitSub) != 0u);
                    const uint64_t slot = sbase + qi;
                    if (slot < p.raw_cap) p.evraw[slot] = make_uint2(c_in, (uint32_t)val);
                    else atomicOr(&p.ctr->flags, kFlagEventOverflow);
                } else if (pos) {
                    // units before k: the low units of words [0, (k+1)/2), the high units of words [0, k/2)
                    p.rd_pre[tf_lo + si] = make_uint2(c_in, xe + events_before(er, k));
                }
            }
            __syncwarp();                                       // qlist is rewritten in the next round
        }
        tf_lo = nf_lo;
        tf_hi = nf_hi;
        g_cur = g_nxt;
        __syncwarp();                                           // every lane is done with stage s
        if (lane == 0) {
            const uint64_t nxt = gwid + (uint64_t)(it + kWarpStages) * stride;
            if (nxt < p.n_wt) {
                fence_proxy_async();
                mbar_expect_tx(&full[s], kBoxBytes);
                tma_load_tile(sm.stage[warp][s], &tmap, (uint32_t)nxt * kRowsPerBox, &full[s], l2_policy);
            }
        }
    }
}

// tile_first[t] = first entry of unit_off[0, n_entries) that is >= t * kWarpTileUnits (n_entries if none), for
// warp tiles t0..t1: the reads that start inside warp tile t are [tile_first[t], tile_first[t+1]).
// Runs when reads are pushed, not per genotyping pass.
__global__ void __launch_bounds__(256)
k_tile_first(const uint64_t *__restrict__ unit_off, uint64_t n_entries, uint64_t t0, uint64_t t1, uint32_t *__restrict__ tile_first)
{
    const uint64_t t = t0 + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t > t1) return;
    const uint64_t target = t * kWarpTileUnits;
    uint64_t lo = 0, hi = n_entries;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (__ldg(unit_off + mid) < target) lo = mid + 1; else hi = mid;
    }
    tile_first[t] = (uint32_t)lo;
}

// ---- encoding at push: one chunk of BAM words -> units (count, exclusive scan of the counts, write)
__global__ void k_unit_count(const uint32_t *__restrict__ words, uint64_t n, uint32_t *__restrict__ cnt)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        cnt[i] = unit_count(words[i]);
}
__global__ void k_unit_write(const uint32_t *__restrict__ words, uint64_t n, const uint32_t *__restrict__ off, uint16_t *__restrict__ out)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        unit_write(words[i], out + off[i]);
}
// unit_off[r] = ubase + off[cig_off[r] - wbase] for reads [r0, r0 + n) whose first word lies in the chunk that starts at
// stream word wbase (off: the chunk's exclusive unit offsets, one past its end included; null: no words at all)
__global__ void k_read_units(const uint64_t *__restrict__ cig_off, uint64_t r0, uint64_t n, uint64_t wbase,
                             const uint32_t *__restrict__ off, uint64_t ubase, uint64_t *__restrict__ unit_off)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        unit_off[r0 + i] = ubase + (off ? off[cig_off[r0 + i] - wbase] : 0u);
}

// Per read: (1) the index of its first event in CIGAR order and the stream-wide consumption prefix
// at its first unit = warp-tile prefix + the tile-local prefix k_cigar_scan left in rd_pre;
// (2) its events moved from warp-tile storage into CIGAR order with absolute anchors:
// pos1 = ref_start + 1 + bases consumed by the read before the op (the u32 cursor of call.rs:380).
// A warp owns 31 reads; lane 31 only supplies the first-event index of the next read.
// `wt` holds EXCLUSIVE prefixes here (k_exclusive_scan2 ran in between).
__global__ void __launch_bounds__(256)
k_read_fixup(const uint64_t *__restrict__ unit_off, const int32_t *__restrict__ rs, uint64_t R,
             const uint2 *__restrict__ wt, const uint2 *__restrict__ rd_pre,
             const uint32_t *__restrict__ wt_sbase, const uint2 *__restrict__ evraw, uint64_t raw_cap,
             uint2 *__restrict__ events, uint64_t ev_cap, uint32_t *__restrict__ ev_off, DevCounters *__restrict__ ctr)
{
    const uint32_t lane = lane_id();
    const uint64_t warp_global = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t r = warp_global * 31 + lane;
    uint32_t e = 0, c = 0;
    uint64_t g = 0;
    if (r <= R) {
        g = unit_off[r];
        const uint2 w0 = wt[g / kWarpTileUnits];
        c = w0.x;
        e = w0.y;
        if (g % kWarpTileUnits) {
            const uint2 pre = rd_pre[r];
            c += pre.x;
            e += pre.y;
        }
    }
    const uint32_t e_next = __shfl_down_sync(0xffffffffu, e, 1);
    if (lane == 31 || r > R) return;
    ev_off[r] = e;
    if (r == R) { ctr->n_events = e; return; }
    if (e == e_next) return;
    const uint32_t base = (uint32_t)rs[r] + 1u - c;
    uint64_t gw = g / kWarpTileUnits;
    uint2 pre = wt[gw];
    uint32_t hi = wt[gw + 1].y;
    for (uint32_t k = e; k < e_next; ++k) {
        while (k >= hi) { ++gw; pre = wt[gw]; hi = wt[gw + 1].y; }
        const uint64_t slot = (uint64_t)wt_sbase[gw] + (k - pre.y);
        if (k < ev_cap && slot < raw_cap) {
            const uint2 raw = evraw[slot];
            events[k] = make_uint2(base + pre.x + raw.x, raw.y);
        } else {
            atomicOr(&ctr->flags, kFlagEventOverflow);
        }
    }
}

// ----------------------------------------------------------------------------------------------
// exclusive scan of u32 counts -> u32 offsets (n+1 outputs), single pass, decoupled look-back
constexpr int kXsThreads = 256;
constexpr int kXsItems = 8;
constexpr int kXsTile = kXsThreads * kXsItems;

__global__ void __launch_bounds__(kXsThreads)
k_exclusive_scan(const uint32_t *in, uint32_t *out, uint64_t n, uint32_t ntiles,
                 uint64_t *__restrict__ desc, unsigned int *__restrict__ tile_counter, unsigned int *__restrict__ overflow_flags)
{
    __shared__ uint32_t wsum[kXsThreads / 32];
    __shared__ uint32_t tile_s;
    __shared__ uint64_t base_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    while (true) {
        if (tid == 0) tile_s = atomicAdd(tile_counter, 1u);
        __syncthreads();
        const uint32_t t = tile_s;
        if (t >= ntiles) break;
        const uint64_t i0 = (uint64_t)t * kXsTile + (uint64_t)tid * kXsItems;
        uint32_t v[kXsItems], sum = 0;
#pragma unroll
        for (int k = 0; k < kXsItems; ++k) {
            v[k] = (i0 + k < n) ? in[i0 + k] : 0u;
            sum += v[k];
        }
        const uint32_t incl = warp_incl_scan(sum);
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        uint32_t wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kXsThreads / 32; ++w) {
            if (w < (int)warp) wbase += wsum[w];
            total += wsum[w];
        }
        if (warp == 0) {
            if (lane == 0) st_relaxed_u64(desc + t, (t == 0 ? kDescPrefix : kDescAggregate) | (uint64_t)total);
            uint64_t base = 0;
            if (t > 0) {
                base = lookback(desc, (int64_t)t);
                if (lane == 0) st_relaxed_u64(desc + t, kDescPrefix | ((base + total) & kDescValueMask));
            }
            if (lane == 0) {
                base_s = base;
                if (t == ntiles - 1) {
                    out[n] = (uint32_t)(base + total);
                    if (overflow_flags && base + total > 0xFFFFFFFFull) atomicOr(overflow_flags, kFlagCountOverflow);
                }
            }
        }
        __syncthreads();
        uint32_t run = (uint32_t)base_s + wbase + incl - sum;
#pragma unroll
        for (int k = 0; k < kXsItems; ++k) {
            if (i0 + k < n) out[i0 + k] = run;
            run += v[k];
        }
        __syncthreads();
    }
}

// same for pairs of u32 (both components wrap mod 2^32; `y` is checked against 2^32): totals `in[0, n)` ->
// exclusive prefixes `out[0, n]`
__global__ void __launch_bounds__(kXsThreads)
k_exclusive_scan2(const uint2 *__restrict__ in, uint2 *__restrict__ out, uint64_t n, uint32_t ntiles,
                  uint64_t *__restrict__ desc_x, uint64_t *__restrict__ desc_y, unsigned int *__restrict__ tile_counter,
                  unsigned int *__restrict__ overflow_flags)
{
    __shared__ uint32_t wsx[kXsThreads / 32], wsy[kXsThreads / 32];
    __shared__ uint32_t tile_s;
    __shared__ uint64_t bx_s, by_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    while (true) {
        if (tid == 0) tile_s = atomicAdd(tile_counter, 1u);
        __syncthreads();
        const uint32_t t = tile_s;
        if (t >= ntiles) break;
        const uint64_t i0 = (uint64_t)t * kXsTile + (uint64_t)tid * kXsItems;
        uint2 v[kXsItems];
        uint32_t sx = 0, sy = 0;
#pragma unroll
        for (int k = 0; k < kXsItems; ++k) {
            v[k] = (i0 + k < n) ? in[i0 + k] : make_uint2(0u, 0u);
            sx += v[k].x;
            sy += v[k].y;
        }
        const uint32_t ix = warp_incl_scan(sx), iy = warp_incl_scan(sy);
        if (lane == 31) { wsx[warp] = ix; wsy[warp] = iy; }
        __syncthreads();
        uint32_t wbx = 0, wby = 0, tx = 0, ty = 0;
#pragma unroll
        for (int w = 0; w < kXsThreads / 32; ++w) {
            if (w < (int)warp) { wbx += wsx[w]; wby += wsy[w]; }
            tx += wsx[w];
            ty += wsy[w];
        }
        if (warp == 0) {
            if (lane == 0) {
                st_relaxed_u64(desc_x + t, (t == 0 ? kDescPrefix : kDescAggregate) | (uint64_t)tx);
                st_relaxed_u64(desc_y + t, (t == 0 ? kDescPrefix : kDescAggregate) | (uint64_t)ty);
            }
            uint64_t bx = 0, by = 0;
            if (t > 0) {
                bx = lookback(desc_x, (int64_t)t);
                by = lookback(desc_y, (int64_t)t);
                if (lane == 0) {
                    st_relaxed_u64(desc_x + t, kDescPrefix | ((bx + tx) & 0xFFFFFFFFull));
                    st_relaxed_u64(desc_y + t, kDescPrefix | ((by + ty) & kDescValueMask));
                }
            }
            if (lane == 0) {
                bx_s = bx;
                by_s = by;
                if (t == ntiles - 1) {
                    out[n] = make_uint2((uint32_t)(bx + tx), (uint32_t)(by + ty));
                    if (overflow_flags && by + ty > 0xFFFFFFFFull) atomicOr(overflow_flags, kFlagCountOverflow);
                }
            }
        }
        __syncthreads();
        uint32_t rx = (uint32_t)bx_s + wbx + ix - sx, ry = (uint32_t)by_s + wby + iy - sy;
#pragma unroll
        for (int k = 0; k < kXsItems; ++k) {
            if (i0 + k < n) out[i0 + k] = make_uint2(rx, ry);
            rx += v[k].x;
            ry += v[k].y;
        }
        __syncthreads();
    }
}

// ----------------------------------------------------------------------------------------------
// K2b: per (read, locus) candidate: the filter (call.rs:297-300 / 350-352), the sum of the read's
// events anchored inside the locus window (call.rs:388,394,400: start < P && P < end) and the
// scatter of the packed call into the locus' segment: H1 (or every unphased call) grows from the
// front of the segment, H2 from its back; one 64-bit atomic per pair hands out the slot.
// The kernel reads the events straight from the scan kernel's warp-tile storage: event k of the stream
// lives in warp tile t with wt[t].y <= k < wt[t+1].y at slot wt_sbase[t] + (k - wt[t].y), and its 1-based
// anchor (the u32 cursor of call.rs:380) is ref_start + 1 + (wt[t].x + raw.x) - (consumption prefix at the
// read's first word).
constexpr int kPairWarps = 4;               // warps per CTA of k_pair_eval (each warp works alone: no block-level sync)
constexpr int kPairMinCtas = 10;            // 40 warps per SM
constexpr int kPairEvPool = 256;            // events per warp (32 consecutive reads) kept in shared memory
constexpr int kPairLociCache = 128;         // catalog entries per warp kept in shared memory
constexpr int kPairTileCache = 64;          // warp-tile prefixes per warp kept in shared memory

struct EventSource {
    const uint64_t *unit_off;     // [R + 1] first unit of every read (+ sentinel)
    const uint2 *wt;              // [n_wt + 1] exclusive prefixes {consumption, events} per warp tile
    const uint2 *rd_pre;          // [R + 1] tile-local prefixes at each read's first unit
    const uint32_t *wt_sbase;     // [n_wt] storage slot of the warp tile's first event
    const uint2 *evraw;           // {consumption inside the warp tile before the op, val}
    uint64_t raw_cap;
};

// stream-wide {consumption, events} prefix at unit g, which is the first unit of read r
__device__ __forceinline__ uint2 read_prefix(const EventSource &es, uint64_t g, uint64_t r)
{
    const uint2 pre = es.rd_pre[r];                          // unconditional: not behind the load of g
    uint2 v = es.wt[g / kWarpTileUnits];
    if (g % kWarpTileUnits) {                               // (rd_pre is only written for reads starting inside a tile)
        v.x += pre.x;
        v.y += pre.y;
    }
    return v;
}

// event k of a read whose words lie in warp tiles [t_lo, t_hi]: {anchor - base, val} via a search in global memory
__device__ __forceinline__ uint2 event_at(const EventSource &es, uint32_t k, uint32_t t_lo, uint32_t t_hi)
{
    while (t_lo < t_hi) {
        const uint32_t mid = (t_lo + t_hi) >> 1;
        if (es.wt[mid + 1].y > k) t_hi = mid; else t_lo = mid + 1;
    }
    const uint2 w = es.wt[t_lo];
    const uint64_t slot = (uint64_t)es.wt_sbase[t_lo] + (k - w.y);
    uint2 raw = make_uint2(0u, 0u);
    if (slot < es.raw_cap) raw = es.evraw[slot];            // (overflowed speculative buffer: the run is repeated)
    return make_uint2(w.x + raw.x, raw.y);
}

// Call keys: 64-bit keys are ((call + 2^61) << 1) | clip with the H2 marker in bit 63. While every call of the reads
// fits 30 bits the pass runs on 32-bit keys of the same layout (bias 2^29, H2 marker in bit 31): half the bytes from
// k_pair_eval to k_locus_median, and half the shuffles and compares of the sorting networks. A call outside that range
// raises kFlagWideCall and the host repeats the pass with 64-bit keys.
template <typename T> struct KeyTraits;
template <> struct KeyTraits<uint64_t> {
    static constexpr uint64_t hap = kKeyHapBit, inf = kKeyInf;
    static __device__ __forceinline__ int64_t call(uint64_t k) { return (int64_t)((k & ~hap) >> 1) - kCallBias; }
};
template <> struct KeyTraits<uint32_t> {
    static constexpr uint32_t hap = 1u << 31, inf = 0xFFFFFFFFu;
    static constexpr int32_t bias = 1 << 29;
    static __device__ __forceinline__ int64_t call(uint32_t k) { return (int64_t)((int32_t)((k & ~hap) >> 1) - bias); }
};

// one read with candidates, as the candidate loop of k_pair_eval reads it: two 16-byte shared-memory loads
struct PairRead {
    uint4 a;                                // rs, re, lo - (flat index of its first candidate), abase
    uint4 b;                                // eb (first staged event), number of events, hf | lane << 16, BAM words
};

struct PairSmem {                           // per CTA of kPairWarps warps (dynamic shared memory)
    uint2 ev[kPairWarps][kPairEvPool];
    PairRead rd[kPairWarps][32];            // the warp's reads with candidates, compacted in lane order
    uint32_t ty[kPairWarps][kPairTileCache + 1], tx[kPairWarps][kPairTileCache], tsb[kPairWarps][kPairTileCache];
    int2 lse[kPairWarps][kPairLociCache];   // start, end
    uint32_t seg[kPairWarps][kPairLociCache + 1];
};

// reads [r_begin, r_end) (the pass launches it once over [0, R); bounding r by rv.R instead doubles ptxas' spills)
// KeyT: uint32_t (calls outside [-2^29, 2^29) raise kFlagWideCall and are not stored) or uint64_t
template <typename KeyT>
__global__ void __launch_bounds__(kPairWarps * 32, kPairMinCtas)
k_pair_eval(ReadView rv, uint64_t r_begin, uint64_t r_end, LocusView lv, int unphased, const uint32_t *__restrict__ cand_lo,
            const uint32_t *__restrict__ cand_n, EventSource es, const uint32_t *__restrict__ seg_off,
            unsigned long long *__restrict__ cursor, KeyT *__restrict__ vals, uint64_t vals_cap,
            DevCounters *__restrict__ ctr)
{
    // A warp owns 32 consecutive reads; their candidates are flattened and dealt to the lanes
    // 32 at a time (reads have 0..hundreds of candidates, a per-read loop leaves most lanes idle).
    // Everything the inner loop needs is staged in shared memory first (the reads' events -- one
    // contiguous run of the event stream, rebased from tile-local to stream-wide consumption on the way
    // in: a read's anchors are its abase + that --, the slice of
    // the catalog the warp touches), so that the only global operations left in the loop are the slot
    // atomic and the store of the call -- and the store is deferred by one iteration so that the atomic's
    // round trip overlaps the next candidate.
    extern __shared__ __align__(16) unsigned char pair_smem_raw[];
    PairSmem &sm = *reinterpret_cast<PairSmem *>(pair_smem_raw);
    auto &s_ev = sm.ev;
    auto &s_ty = sm.ty; auto &s_tx = sm.tx; auto &s_tsb = sm.tsb; auto &s_lse = sm.lse; auto &s_seg = sm.seg;
    const uint32_t lane = lane_id(), wid = threadIdx.x >> 5;
    const uint64_t r = r_begin + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    uint32_t n = 0, lo = 0, e0 = 0xFFFFFFFFu, e1 = 0xFFFFFFFFu, hf = 0, words = 0, t_lo = 0, t_hi = 0, abase = 0;
    int32_t rs = 0, re = 0;
    if (r < r_end) {
        // independent loads, all in flight together
        n = cand_n[r];
        lo = cand_lo[r];
        rs = rv.rs[r];
        re = rv.re[r];
        hf = (uint32_t)rv.hp[r] | ((uint32_t)(rv.flags[r] & 1u) << 8) | ((uint32_t)(rv.flags[r] & 2u) << 9);   // bit 10: SA panic
        const uint64_t g0 = es.unit_off[r], g1 = es.unit_off[r + 1];
        const uint2 p0 = read_prefix(es, g0, r), p1 = read_prefix(es, g1, r + 1);
        e0 = p0.y;
        e1 = p1.y;
        abase = (uint32_t)rs + 1u - p0.x;                       // anchor = abase + stream-wide consumption before the op
        t_lo = (uint32_t)(g0 / kWarpTileUnits);
        t_hi = g1 > g0 ? (uint32_t)((g1 - 1) / kWarpTileUnits) : t_lo;
        words = (uint32_t)min(rv.cig_off[r + 1] - rv.cig_off[r], (uint64_t)0xFFFFFFFFu);   // BAM words: the statistics
    }
    // the events of the warp's joined reads are one run [ev_lo, ev_hi) of the event stream, stored in the
    // warp tiles [tile_lo, tile_hi]; the tile range only depends on unit_off, so its prefixes are fetched
    // while the per-read prefixes are still in flight
    const uint32_t tile_lo = __reduce_min_sync(0xffffffffu, n ? t_lo : 0xFFFFFFFFu);
    const uint32_t tile_hi = __reduce_max_sync(0xffffffffu, n ? t_hi : 0u);
    const uint32_t nt = tile_hi - tile_lo + 1u;
    const bool tiles_cached = tile_lo <= tile_hi && nt <= (uint32_t)kPairTileCache;
    if (tiles_cached) {
        for (uint32_t i = lane; i <= nt; i += 32) {
            const uint2 w = es.wt[tile_lo + i];
            s_ty[wid][i] = w.y;
            if (i < nt) {
                s_tx[wid][i] = w.x;
                s_tsb[wid][i] = es.wt_sbase[tile_lo + i];
            }
        }
    }
    const uint32_t ev_lo = __reduce_min_sync(0xffffffffu, n ? e0 : 0xFFFFFFFFu);
    const uint32_t ev_hi = __reduce_max_sync(0xffffffffu, n ? e1 : 0u);
    __syncwarp();
    if (ev_lo < ev_hi) {
        const uint32_t cnt = min(ev_hi - ev_lo, (uint32_t)kPairEvPool);
        // pass 1: where each event lives (storage slot) and the consumption prefix of its tile -- parked in s_ev
        // (enumerating the events tile by tile instead was measured: fewer instructions, but 14 dependent shared-memory
        // round trips in a row per warp -- 0.57 ms instead of 0.52 for the kernel)
        uint32_t ta = 0;                                        // cached tiles: this lane's k only grows, so does its tile
        for (uint32_t i = lane; i < cnt; i += 32) {
            const uint32_t k = ev_lo + i;
            uint32_t slot, rel;                                 // rel: stream-wide consumption before the tile
            if (tiles_cached) {
                // first tile t with ty[t + 1] > k: 32 events further on is typically 2-3 tiles further on
                while (ta + 1u < nt && s_ty[wid][ta + 1u] <= k) ++ta;
                slot = s_tsb[wid][ta] + (k - s_ty[wid][ta]);
                rel = s_tx[wid][ta];
            } else {
                uint32_t a = tile_lo, b = tile_hi;
                while (a < b) {
                    const uint32_t mid = (a + b) >> 1;
                    if (es.wt[mid + 1].y > k) b = mid; else a = mid + 1;
                }
                const uint2 w = es.wt[a];
                slot = es.wt_sbase[a] + (k - w.y);
                rel = w.x;
            }
            s_ev[wid][i] = make_uint2(slot, rel);
        }
        // pass 2: independent loads from the event storage (several in flight per lane)
#pragma unroll 4
        for (uint32_t i = lane; i < cnt; i += 32) {
            const uint2 sr = s_ev[wid][i];
            uint2 raw = make_uint2(0u, 0u);
            if ((uint64_t)sr.x < es.raw_cap) raw = es.evraw[sr.x];   // (overflowed speculative buffer: the run is repeated)
            s_ev[wid][i] = make_uint2(sr.y + raw.x, raw.y);
        }
    }
    if (n && e1 - ev_lo > (uint32_t)kPairEvPool) hf |= 1u << 9;      // not (entirely) staged: searched in global memory
    const uint32_t incl = warp_incl_scan(n);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t off = incl - n;                                    // flat index of the read's first candidate
    // the record of a read with candidates goes to its rank among them: the loop below finds the read of a candidate by
    // counting the reads that start in front of it (reads without candidates start nowhere)
    const uint32_t with_cands = __ballot_sync(0xffffffffu, n != 0);
    if (n) {
        sm.rd[wid][__popc(with_cands & lanemask_lt())] =
            PairRead{make_uint4((uint32_t)rs, (uint32_t)re, lo - off, abase), make_uint4(e0 - ev_lo, e1 - e0, hf | (lane << 16), words)};
    }
    // slice of the catalog this warp touches
    const uint32_t lo_min = __reduce_min_sync(0xffffffffu, n ? lo : 0xFFFFFFFFu);
    const uint32_t hi_max = __reduce_max_sync(0xffffffffu, n ? lo + n : 0u);
    const bool cached = total && (hi_max - lo_min <= (uint32_t)kPairLociCache);
    if (cached) {
        const uint32_t span = hi_max - lo_min;
        for (uint32_t i = lane; i < span; i += 32) {
            s_lse[wid][i] = make_int2(__ldg(lv.start + lo_min + i), __ldg(lv.end + lo_min + i));
        }
        for (uint32_t i = lane; i <= span; i += 32) s_seg[wid][i] = __ldg(seg_off + lo_min + i);
    }
    __syncwarp();

    uint32_t npass = 0;                 // pairs that land in a bucket
    uint32_t joined_bits = 0;           // lanes of the warp whose reads had a pair land here
    uint64_t visits = 0;                // CIGAR words the reference walks: every passing pair, incl. HP 0
    bool bad_hp = false, bad_sa = false;
    // deferred store of the previous candidate
    bool pend = false, wide = false;
    unsigned long long pend_old = 0;
    KeyT pend_key = 0;
    uint32_t pend_seg = 0, pend_cap = 0;
    bool pend_back = false;
    auto flush_pending = [&]() {
        if (!pend) return;
        const uint32_t slot_k = pend_back ? (uint32_t)(pend_old >> 32) : (uint32_t)pend_old;
        const uint64_t slot = pend_back ? (uint64_t)pend_seg + (pend_cap - 1u - slot_k) : (uint64_t)pend_seg + slot_k;
        if (slot_k < pend_cap && slot < vals_cap) vals[slot] = pend_key;
        else atomicOr(&ctr->flags, kFlagValsOverflow);
        pend = false;
    };

    uint32_t owner = 0xFFFFFFFFu;       // rank of the read that owns flat index base - 1
    for (uint32_t base = 0; base < total; base += 32) {
        const uint32_t k = base + lane;
        const bool active = k < total;
        // owning read: the reads starting in [base, base + 32) as a bit mask over the positions, counted up to k
        const uint32_t starts = __reduce_or_sync(0xffffffffu, (n && off - base < 32u) ? 1u << (off - base) : 0u);
        const PairRead &pr = sm.rd[wid][owner + __popc(starts & lanemask_le())];
        owner += __popc(starts);
        const uint4 ra = pr.a, rb = pr.b;
        const int32_t rs_j = (int32_t)ra.x, re_j = (int32_t)ra.y;
        const uint32_t abase_j = ra.w, eb_j = rb.x, ne_j = rb.y, hf_j = rb.z & 0xFFFFu, j = rb.z >> 16;
        bool emit = false;
        uint32_t l = 0, h = 0, seg = 0, cap = 0;
        int32_t ls = 0, le = 0;
        if (active) {
            l = k + ra.z;
            h = hf_j & 0xFFu;
            if (cached) {
                const int2 se = s_lse[wid][l - lo_min];
                ls = se.x;
                le = se.y;
                seg = s_seg[wid][l - lo_min];
                cap = s_seg[wid][l - lo_min + 1] - seg;
            } else {
                ls = __ldg(lv.start + l);
                le = __ldg(lv.end + l);
                seg = __ldg(seg_off + l);
                cap = __ldg(seg_off + l + 1) - seg;
            }
            if (pair_passes(unphased != 0, rs_j, re_j, ls, le)) {
                visits += rb.w;                             // call.rs:357 runs before the bucket lookup
                emit = true;
                if (hf_j & (1u << 10)) {                    // call.rs:394 -> 431: the walk panics inside is_accidental_2d
                    bad_sa = true;
                    ctr->bad_sa_read = r - lane + j;
                    emit = false;
                } else if (!unphased) {
                    if (h > 2u) {                           // call.rs:358 unwrap on None
                        bad_hp = true;
                        ctr->bad_hp_value = h;
                        ctr->bad_hp_read = r - lane + j;
                        emit = false;
                    } else if (h == 0u) {
                        emit = false;                       // HP 0 lands in the ignored bucket
                    }
                }
            }
        }
        unsigned long long old = 0;
        KeyT key = 0;
        const bool back = !unphased && h == 2u;
        if (emit) {
            ++npass;
            joined_bits |= 1u << j;
            // slot first: the atomic's round trip overlaps the rest of this iteration and the next one
            old = atomicAdd(cursor + l, back ? (1ull << 32) : 1ull);
            const uint32_t start_ext = (uint32_t)ls - 10u, end_ext = (uint32_t)le + 10u;
            const bool is2d = ((hf_j >> 8) & 1u) != 0u;
            int64_t call = 0;
            uint32_t clip = 0;
            if (!(hf_j & (1u << 9))) {
                // the read's events sit in shared memory, sorted by anchor: binary search, then a short scan
                const uint32_t ne = ne_j;
                const uint2 *sev = &s_ev[wid][eb_j];
                uint32_t a = 0, b = ne;
                while (a < b) {
                    const uint32_t m = (a + b) >> 1;
                    if (abase_j + sev[m].x > start_ext) b = m; else a = m + 1;
                }
                for (uint32_t q = a; q < ne; ++q) {
                    const uint2 ev = sev[q];
                    if (!(abase_j + ev.x < end_ext)) break; // start_ext < P && P < end_ext (call.rs:388,394,400)
                    const int32_t v = (int32_t)ev.y;
                    const uint32_t is_s = (uint32_t)v & 1u;
                    if (is_s && is2d) continue;             // call.rs:394 !is_accidental_2d(&r)
                    call += (int64_t)(v >> 1);
                    clip |= is_s;
                }
            } else {
                // long event list, read from the warp-tile storage: anchors increase along the read, so a
                // binary search finds the first event with pos1 > start_ext; then a short scan. The tile search runs over
                // the warp's tiles: they hold the read's, and the tile of an event is the same over any range that does
                const uint32_t e0_j = ev_lo + eb_j, e1_j = e0_j + ne_j;
                uint32_t a = e0_j, b = e1_j;
                while (a < b) {
                    const uint32_t m = (a + b) >> 1;
                    if (abase_j + event_at(es, m, tile_lo, tile_hi).x > start_ext) b = m; else a = m + 1;
                }
                for (uint32_t e = a; e < e1_j; ++e) {
                    const uint2 ev = event_at(es, e, tile_lo, tile_hi);
                    if (!(abase_j + ev.x < end_ext)) break;
                    const int32_t v = (int32_t)ev.y;
                    const uint32_t is_s = (uint32_t)v & 1u;
                    if (is_s && is2d) continue;             // call.rs:394 !is_accidental_2d(&r)
                    call += (int64_t)(v >> 1);
                    clip |= is_s;
                }
            }
            if constexpr (sizeof(KeyT) == 8) {
                key = ((uint64_t)(call + kCallBias) << 1) | clip;
            } else if (call >= -(int64_t)KeyTraits<uint32_t>::bias && call < (int64_t)KeyTraits<uint32_t>::bias) {
                key = ((uint32_t)(call + KeyTraits<uint32_t>::bias) << 1) | clip;
            } else {
                wide = true;                                // the slot stays taken and unwritten: the pass is repeated
                emit = false;
            }
        }
        flush_pending();                                    // store of the previous candidate
        if (emit) {
            pend = true;
            pend_old = old;
            pend_key = key;
            pend_seg = seg;
            pend_cap = cap;
            pend_back = back;
        }
    }
    flush_pending();
    __syncwarp();
    // statistics (one atomic per warp per counter)
    const bool joined = ((__reduce_or_sync(0xffffffffu, joined_bits) >> lane) & 1u) != 0u;
    const uint32_t pass_w = __reduce_add_sync(0xffffffffu, npass);
    const uint32_t join_w = __popc(__ballot_sync(0xffffffffu, joined));
    const uint64_t words_w = warp_sum(joined ? (uint64_t)words : 0ull);
    const uint64_t visits_w = warp_sum(visits);
    const uint32_t bad_w = __any_sync(0xffffffffu, bad_hp), bad_sa_w = __any_sync(0xffffffffu, bad_sa);
    const uint32_t wide_w = __any_sync(0xffffffffu, wide);
    if (lane == 0) {
        // one of kStatSlots copies per warp: no block barrier, and no single hot address in L2
        unsigned long long *slot = ctr->stat[(blockIdx.x * (uint32_t)kPairWarps + wid) % kStatSlots];
        if (pass_w) atomicAdd(slot + ST_PAIRS, (unsigned long long)pass_w);
        if (join_w) atomicAdd(slot + ST_READS_JOINED, (unsigned long long)join_w);
        if (words_w) atomicAdd(slot + ST_WORDS_JOINED, (unsigned long long)words_w);
        if (visits_w) atomicAdd(slot + ST_OP_VISITS, (unsigned long long)visits_w);
        if (bad_w) atomicOr(&ctr->flags, kFlagBadHp);
        if (bad_sa_w) atomicOr(&ctr->flags, kFlagBadSa);
        if (wide_w) atomicOr(&ctr->flags, kFlagWideCall);
    }
}

// ----------------------------------------------------------------------------------------------
// K3: per-locus sort / split / support filter / median (call.rs:308-321,365-369,497-522).
// Keys are 63-bit ((call + bias) << 1 | clip): ascending key order == (value, Span before Clip).
// Phased loci set bit 63 on H2 keys so one sort orders [H1 | H2]; unphased loci split the sorted
// run at n/2 (call.rs:314).

// all-ascending bitonic network over K striped registers per lane (element i = k*32 + lane)
// N < K * 32 sorts every aligned run of N elements on its own
template <int K, typename T, int N = K * 32>
__device__ __forceinline__ void warp_sort(T (&key)[K])
{
#pragma unroll
    for (int blk = 2; blk <= N; blk <<= 1) {
        // mirror step: partner = i ^ (blk - 1)
        {
            const int lane_x = (blk - 1) & 31, reg_x = (blk - 1) >> 5;
            T other[K];
#pragma unroll
            for (int k = 0; k < K; ++k) other[k] = __shfl_xor_sync(0xffffffffu, key[k ^ reg_x], lane_x);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int i = k * 32 + (int)lane_id();
                const bool lower = (i & (blk >> 1)) == 0;      // lower half of the mirrored block keeps the min
                const T a = key[k], b = other[k];
                key[k] = lower ? (a < b ? a : b) : (a > b ? a : b);
            }
        }
#pragma unroll
        for (int d = blk >> 2; d >= 1; d >>= 1) {
            const int lane_x = d & 31, reg_x = d >> 5;
            T other[K];
#pragma unroll
            for (int k = 0; k < K; ++k)
                other[k] = lane_x ? __shfl_xor_sync(0xffffffffu, key[k ^ reg_x], lane_x) : key[k ^ reg_x];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int i = k * 32 + (int)lane_id();
                const bool lower = (i & d) == 0;
                const T a = key[k], b = other[k];
                key[k] = lower ? (a < b ? a : b) : (a > b ? a : b);
            }
        }
    }
}

__device__ __forceinline__ int64_t key_call(uint64_t key) { return KeyTraits<uint64_t>::call(key); }

// median of the sorted sub-range [a, a+n) held striped across the warp. Returns validity;
// *twice = 2 x median. call.rs:497-522.
template <int K, typename T>
__device__ __forceinline__ bool warp_median_part(const T (&key)[K], uint32_t a, uint32_t n, uint32_t support,
                                                 int64_t *twice, bool *panicked)
{
    *twice = 0;
    if (n < support) return false;                                   // call.rs:498-500
    uint32_t span_b[K], clip_b[K];
    uint32_t s = 0, c = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t i = k * 32 + lane_id();
        const bool in = (i >= a) && (i < a + n);
        span_b[k] = __ballot_sync(0xffffffffu, in && !(key[k] & 1u));
        clip_b[k] = __ballot_sync(0xffffffffu, in && (key[k] & 1u));
        s += __popc(span_b[k]);
        c += __popc(clip_b[k]);
    }
    const uint32_t topk = (s <= support) ? (support - s) : 0u;       // call.rs:509-513
    const uint32_t m = s + topk;
    if (m == 0) { *panicked = true; return false; }                  // call.rs:516 on an empty vector
    const uint32_t t2 = m >> 1, t1 = (m & 1u) ? t2 : t2 - 1u;        // call.rs:515-521
    uint32_t clip_before = 0, sel_before = 0;
    int64_t sum = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t me = 1u << lane_id();
        const bool is_span = (span_b[k] & me) != 0, is_clip = (clip_b[k] & me) != 0;
        const uint32_t clip_idx = clip_before + __popc(clip_b[k] & lanemask_lt());
        const bool sel = is_span || (is_clip && clip_idx + topk >= c);   // the topk largest clips
        const uint32_t sel_b = __ballot_sync(0xffffffffu, sel);
        const uint32_t rank = sel_before + __popc(sel_b & lanemask_lt());
        if (sel) {
            const int64_t v = KeyTraits<T>::call(key[k]);
            if (rank == t1) sum += v;
            if (rank == t2) sum += v;
        }
        clip_before += __popc(clip_b[k]);
        sel_before += __popc(sel_b);
    }
    // (handing the two middle keys out by ballot + shuffle instead was measured: 15 % slower)
    *twice = warp_sum(sum);
    return true;
}

// A locus' segment [seg, seg+cap) holds its H1 calls at the front and its H2 calls at the back
// (unphased: everything at the front). nf/nb = number of front/back entries; n1 = split point of
// the sorted run (phased: nf, unphased: (nf)/2).
// Both haplotypes of a phased locus in one pass (call.rs:497-522 twice): 32-bit keys, H1 sorted in lanes
// 0-15 (nf of them), H2 sorted in lanes 16-31 (nb of them). Every lane works on its own half: the ballots
// are shared, the counts are taken under the half's lane mask.
__device__ __forceinline__ void median_halves32(uint32_t key, uint32_t nf, uint32_t nb, uint32_t support, int64_t *t1,
                                                int64_t *t2, uint32_t *valid, bool *panicked)
{
    const uint32_t lane = lane_id();
    const bool upper = lane >= 16u;
    const uint32_t hm = upper ? 0xFFFF0000u : 0x0000FFFFu;
    const uint32_t n = upper ? nb : nf;
    const bool in = (lane & 15u) < n;
    const uint32_t span_b = __ballot_sync(0xffffffffu, in && !(key & 1u));
    const uint32_t clip_b = __ballot_sync(0xffffffffu, in && (key & 1u));
    const uint32_t s = __popc(span_b & hm), c = __popc(clip_b & hm);
    const bool enough = n >= support;                                // call.rs:498-500
    const uint32_t topk = (s <= support) ? (support - s) : 0u;       // call.rs:509-513
    const uint32_t m = s + topk;
    const bool ok = enough && m != 0u;                               // m == 0: call.rs:516 on an empty vector
    const uint32_t i2 = m >> 1, i1 = (m & 1u) ? i2 : i2 - 1u;        // call.rs:515-521
    const uint32_t below = hm & lanemask_lt();
    const bool is_span = (span_b >> lane) & 1u, is_clip = (clip_b >> lane) & 1u;
    const bool sel = ok && (is_span || (is_clip && __popc(clip_b & below) + topk >= c));   // the topk largest clips
    const uint32_t sel_b = __ballot_sync(0xffffffffu, sel);
    const uint32_t rank = __popc(sel_b & below);
    int32_t sum = 0;                                                 // |call| < 2^29: two of them fit
    if (sel) {
        const int32_t v = (int32_t)KeyTraits<uint32_t>::call(key);
        sum = (rank == i1 ? v : 0) + (rank == i2 ? v : 0);
    }
#pragma unroll
    for (int d = 8; d >= 1; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    const uint32_t ok_b = __ballot_sync(0xffffffffu, ok), bad_b = __ballot_sync(0xffffffffu, enough && m == 0u);
    *t1 = (ok_b & 1u) ? (int64_t)__shfl_sync(0xffffffffu, sum, 0) : 0;
    *t2 = (ok_b & 0x10000u) ? (int64_t)__shfl_sync(0xffffffffu, sum, 16) : 0;
    *valid = ((ok_b & 1u) ? 1u : 0u) | ((ok_b & 0x10000u) ? 2u : 0u);
    if (bad_b & 0x10001u) *panicked = true;
}

// kSplit > 0 (phased only): H1 lives at positions [0, nf) and H2 at [kSplit, kSplit + nb) and the two
// runs of kSplit elements are sorted independently (a shorter network than one sort over both).
// 32-bit keys are sorted as they are; 64-bit keys are narrowed to 32 bits where every call of the locus fits.
template <int K, int kSplit, typename KeyT>
__device__ __forceinline__ void warp_locus(const KeyT *__restrict__ vals, uint32_t seg, uint32_t cap, uint32_t nf,
                                           uint32_t nb, uint32_t n1, bool phased, uint32_t support, int64_t *t1,
                                           int64_t *t2, uint32_t *valid, bool *panicked)
{
    const uint32_t ntot = nf + nb;
    constexpr int kSortN = kSplit ? kSplit : K * 32;
    const uint32_t a2 = kSplit ? (uint32_t)kSplit : n1;              // first position of the second part
    if constexpr (sizeof(KeyT) == 4) {
        uint32_t k32[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t i = k * 32 + lane_id();
            uint32_t v = KeyTraits<uint32_t>::inf;
            if constexpr (kSplit > 0) {
                if (i < nf) v = vals[seg + i];
                else if (i >= (uint32_t)kSplit && i - (uint32_t)kSplit < nb) v = vals[seg + cap - nb + (i - (uint32_t)kSplit)];
            } else {
                if (i < nf) v = vals[seg + i];
                else if (i < ntot) v = vals[seg + cap - nb + (i - nf)] | (phased ? KeyTraits<uint32_t>::hap : 0u);
            }
            k32[k] = v;
        }
        warp_sort<K, uint32_t, kSortN>(k32);
        if constexpr (K == 1 && kSplit == 16) {
            median_halves32(k32[0], nf, nb, support, t1, t2, valid, panicked);
        } else {
            const bool v1 = warp_median_part<K, uint32_t>(k32, 0, n1, support, t1, panicked);
            const bool v2 = warp_median_part<K, uint32_t>(k32, a2, ntot - n1, support, t2, panicked);
            *valid = (v1 ? 1u : 0u) | (v2 ? 2u : 0u);
        }
        return;
    }
    uint64_t key[K];
    bool have_k[K];
    bool small = true;                      // every call fits the 32-bit key layout
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t i = k * 32 + lane_id();
        uint64_t v = kKeyInf;
        bool have;
        if constexpr (kSplit > 0) {
            have = (i < nf) || (i >= (uint32_t)kSplit && i - (uint32_t)kSplit < nb);
            if (i < nf) v = (uint64_t)vals[seg + i];
            else if (have) v = (uint64_t)vals[seg + cap - nb + (i - (uint32_t)kSplit)];
        } else {
            have = i < ntot;
            if (i < nf) v = (uint64_t)vals[seg + i];
            else if (have) v = (uint64_t)vals[seg + cap - nb + (i - nf)] | (phased ? kKeyHapBit : 0ull);
        }
        if (have) {
            const int64_t c = key_call(v);
            small = small && c >= -(int64_t)KeyTraits<uint32_t>::bias && c < (int64_t)KeyTraits<uint32_t>::bias;
        }
        key[k] = v;
        have_k[k] = have;
    }
    bool v1, v2;
    if (__all_sync(0xffffffffu, small)) {
        uint32_t k32[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint64_t v = key[k];
            const uint32_t body = (uint32_t)((key_call(v) + KeyTraits<uint32_t>::bias) << 1) | (uint32_t)(v & 1ull);
            k32[k] = have_k[k] ? (body | ((v & kKeyHapBit) ? KeyTraits<uint32_t>::hap : 0u)) : KeyTraits<uint32_t>::inf;
        }
        warp_sort<K, uint32_t, kSortN>(k32);
        if constexpr (K == 1 && kSplit == 16) {
            median_halves32(k32[0], nf, nb, support, t1, t2, valid, panicked);
            return;
        }
        v1 = warp_median_part<K, uint32_t>(k32, 0, n1, support, t1, panicked);
        v2 = warp_median_part<K, uint32_t>(k32, a2, ntot - n1, support, t2, panicked);
    } else {
        warp_sort<K, uint64_t, kSortN>(key);
        v1 = warp_median_part<K, uint64_t>(key, 0, n1, support, t1, panicked);
        v2 = warp_median_part<K, uint64_t>(key, a2, ntot - n1, support, t2, panicked);
    }
    *valid = (v1 ? 1u : 0u) | (v2 ? 2u : 0u);
}

constexpr int kMedianWarpMax = 128;         // loci with more calls go to the CTA kernel
constexpr int kMedianMinCtas = 8;

// header of one locus' segment
struct LocusSeg {
    uint32_t seg, cap, nf, nb;
    bool ok;
};
__device__ __forceinline__ LocusSeg locus_seg(uint32_t seg, uint32_t cap, unsigned long long cur, uint64_t vals_cap)
{
    LocusSeg h;
    h.seg = seg;
    h.cap = cap;
    h.ok = (uint64_t)seg + cap <= vals_cap;
    h.nf = min((uint32_t)cur, cap);
    h.nb = min((uint32_t)(cur >> 32), cap - h.nf);
    return h;
}
// the common phased case (both haplotypes <= 16 calls): lane i < 16 holds H1's call i, lane 16 + i H2's call i
template <typename KeyT>
__device__ __forceinline__ KeyT fast16_load(const KeyT *__restrict__ vals, const LocusSeg &h)
{
    const uint32_t i = lane_id();
    if (i < h.nf) return vals[h.seg + i];
    if (i >= 16u && i - 16u < h.nb) return vals[h.seg + h.cap - h.nb + (i - 16u)];
    return KeyTraits<KeyT>::inf;
}

// one locus: everything after the header. `pre`: the keys of the fast path, already loaded (inf lanes are empty).
template <typename KeyT>
__device__ __forceinline__ void median_one(uint32_t l, uint32_t l0, int chunk, int unphased, uint32_t support, const LocusSeg &h, bool fast, KeyT pre,
                                           const KeyT *__restrict__ vals, int64_t *__restrict__ twice_h1, int64_t *__restrict__ twice_h2,
                                           uint8_t *__restrict__ valid, uint32_t *__restrict__ big_list, DevCounters *__restrict__ ctr)
{
    if (!h.ok) {                                        // speculatively sized call buffer too small: the run is repeated
        if (lane_id() == 0) atomicOr(&ctr->flags, kFlagValsOverflow);
        return;
    }
    const uint32_t nf = h.nf, nb = h.nb, seg = h.seg, cap = h.cap;
    const uint32_t ntot = nf + nb;
    const uint32_t n1 = unphased ? (ntot >> 1) : nf;               // call.rs:314 split_at(len/2)
    int64_t t1 = 0, t2 = 0;
    uint32_t vm = 0;
    bool panicked = false;
    bool done = false;
    if constexpr (sizeof(KeyT) == 4) {
        if (fast) {                                     // keys are here already
            uint32_t k32[1] = {pre};
            warp_sort<1, uint32_t, 16>(k32);
            median_halves32(k32[0], nf, nb, support, &t1, &t2, &vm, &panicked);
            done = true;
        }
    } else if (fast) {
        // keys are here already: 32-bit layout when every call fits 30 bits (practically always)
        const bool have = pre != kKeyInf;
        const int64_t c = key_call(pre);
        const bool small = !have || (c >= -(int64_t)KeyTraits<uint32_t>::bias && c < (int64_t)KeyTraits<uint32_t>::bias);
        if (__all_sync(0xffffffffu, small)) {
            uint32_t k32[1];
            k32[0] = have ? ((uint32_t)((c + KeyTraits<uint32_t>::bias) << 1) | (uint32_t)(pre & 1ull)) : KeyTraits<uint32_t>::inf;
            warp_sort<1, uint32_t, 16>(k32);
            median_halves32(k32[0], nf, nb, support, &t1, &t2, &vm, &panicked);
            done = true;
        }
    }
    if (!done) {
        if (!unphased && nf <= 16 && nb <= 16) warp_locus<1, 16, KeyT>(vals, seg, cap, nf, nb, n1, true, support, &t1, &t2, &vm, &panicked);
        else if (ntot <= 32) warp_locus<1, 0, KeyT>(vals, seg, cap, nf, nb, n1, !unphased, support, &t1, &t2, &vm, &panicked);
        else if (!unphased && nf <= 32 && nb <= 32) warp_locus<2, 32, KeyT>(vals, seg, cap, nf, nb, n1, true, support, &t1, &t2, &vm, &panicked);
        else if (ntot <= 64) warp_locus<2, 0, KeyT>(vals, seg, cap, nf, nb, n1, !unphased, support, &t1, &t2, &vm, &panicked);
        else if (ntot <= kMedianWarpMax) warp_locus<4, 0, KeyT>(vals, seg, cap, nf, nb, n1, !unphased, support, &t1, &t2, &vm, &panicked);
        else {
            if (lane_id() == 0) big_list[l0 + atomicAdd(&ctr->big_count[chunk], 1u)] = l;
            return;
        }
    }
    if (lane_id() == 0) {
        twice_h1[l] = t1;
        twice_h2[l] = t2;
        valid[l] = (uint8_t)vm;
        if (panicked) atomicOr(&ctr->flags, kFlagMedianEmpty);
    }
}

// A warp owns one locus. Each locus costs two dependent round trips (segment header, then its calls). Warps that took
// several loci, with all headers and then all key loads in flight together before any locus was reduced, were measured
// and do not pay: 1 locus -> 0.357 ms, 2 -> 0.369-0.389, 3 -> 0.473. The kernel is issue-bound, not latency-bound: 68 %
// of the issue slots are busy already and the extra registers cost occupancy.
template <typename KeyT>
__global__ void __launch_bounds__(256, kMedianMinCtas)
k_locus_median(uint32_t l0, uint32_t l1, int chunk, int unphased, uint32_t support, const uint32_t *__restrict__ seg_off,
               const unsigned long long *__restrict__ cursor, const KeyT *__restrict__ vals, uint64_t vals_cap,
               int64_t *__restrict__ twice_h1, int64_t *__restrict__ twice_h2, uint8_t *__restrict__ valid,
               uint32_t *__restrict__ big_list, DevCounters *__restrict__ ctr)
{
    // loci [l0, l1) of the catalog (chunk < kMaxMedianChunks); the chunk's CTA-path loci are listed in big_list[l0 ...]
    const uint32_t l = l0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (l >= l1) return;
    // round trip 1: the header
    const uint32_t seg = seg_off[l], seg_end = seg_off[l + 1];
    const LocusSeg h = locus_seg(seg, seg_end - seg, cursor[l], vals_cap);
    // round trip 2: the calls, on the common path
    const bool fast = h.ok && !unphased && h.nf <= 16u && h.nb <= 16u;
    const KeyT pre = fast ? fast16_load(vals, h) : KeyTraits<KeyT>::inf;
    median_one(l, l0, chunk, unphased, support, h, fast, pre, vals, twice_h1, twice_h2, valid, big_list, ctr);
}

// CTA-wide path for loci with more than kMedianWarpMax calls: bitonic sort in shared memory when
// the run fits, otherwise in place in the (scratch) vals array; then a block-wide selection pass.
constexpr int kBigThreads = 256;
constexpr int kBigSmemKeys = 4096;

template <typename KeyT>
__device__ __forceinline__ void block_part_median(volatile KeyT *a, uint32_t lo, uint32_t n, uint32_t support,
                                                  int64_t *twice, bool *ok, bool *panicked, uint32_t *sh_cnt,
                                                  unsigned long long *sh_acc)
{
    // sh_cnt[0..1]: spans, clips ; sh_cnt[2]: running selected count ; sh_acc: sum of the median elements
    const uint32_t tid = threadIdx.x;
    *twice = 0;
    *ok = false;
    if (n < support) return;
    if (tid == 0) { sh_cnt[0] = 0; sh_cnt[1] = 0; sh_cnt[2] = 0; sh_cnt[3] = 0; *sh_acc = 0ull; }
    __syncthreads();
    uint32_t my_s = 0, my_c = 0;
    for (uint32_t i = tid; i < n; i += blockDim.x) {
        if (a[lo + i] & 1u) ++my_c; else ++my_s;
    }
    my_s = warp_sum(my_s);
    my_c = warp_sum(my_c);
    if (lane_id() == 0) { atomicAdd(&sh_cnt[0], my_s); atomicAdd(&sh_cnt[1], my_c); }
    __syncthreads();
    const uint32_t s = sh_cnt[0], c = sh_cnt[1];
    const uint32_t topk = (s <= support) ? (support - s) : 0u;
    const uint32_t m = s + topk;
    if (m == 0) { *panicked = true; return; }
    const uint32_t t2 = m >> 1, t1 = (m & 1u) ? t2 : t2 - 1u;
    __shared__ uint32_t wtot[2][kBigThreads / 32];
    // chunked pass in sorted order; running counts of clips (sh_cnt[3]) and selected (sh_cnt[2])
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        const uint32_t i = base + tid;
        const bool in = i < n;
        const KeyT k = in ? a[lo + i] : (KeyT)0;
        const bool is_clip = in && (k & 1u), is_span = in && !(k & 1u);
        const uint32_t cb = __ballot_sync(0xffffffffu, is_clip);
        if (lane_id() == 0) wtot[0][tid >> 5] = __popc(cb);
        __syncthreads();
        uint32_t clip_idx = sh_cnt[3] + __popc(cb & lanemask_lt());
        for (uint32_t w = 0; w < (tid >> 5); ++w) clip_idx += wtot[0][w];
        const bool sel = is_span || (is_clip && clip_idx + topk >= c);
        const uint32_t sb = __ballot_sync(0xffffffffu, sel);
        if (lane_id() == 0) wtot[1][tid >> 5] = __popc(sb);
        __syncthreads();
        uint32_t rank = sh_cnt[2] + __popc(sb & lanemask_lt());
        for (uint32_t w = 0; w < (tid >> 5); ++w) rank += wtot[1][w];
        if (sel) {
            const int64_t v = KeyTraits<KeyT>::call(k);
            if (rank == t1) atomicAdd(sh_acc, (unsigned long long)v);
            if (rank == t2) atomicAdd(sh_acc, (unsigned long long)v);
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t ct = 0, st = 0;
            for (uint32_t w = 0; w < blockDim.x / 32; ++w) { ct += wtot[0][w]; st += wtot[1][w]; }
            sh_cnt[3] += ct;
            sh_cnt[2] += st;
        }
        __syncthreads();
    }
    *twice = (int64_t)*sh_acc;
    *ok = true;
}

template <typename KeyT>
__global__ void __launch_bounds__(kBigThreads)
k_locus_median_big(uint32_t l0, int chunk, int unphased, uint32_t support, const uint32_t *__restrict__ seg_off,
                   const unsigned long long *__restrict__ cursor, KeyT *__restrict__ vals, uint64_t vals_cap,
                   int64_t *__restrict__ twice_h1, int64_t *__restrict__ twice_h2, uint8_t *__restrict__ valid,
                   const uint32_t *__restrict__ big_list, DevCounters *__restrict__ ctr)
{
    constexpr KeyT hap = KeyTraits<KeyT>::hap, inf = KeyTraits<KeyT>::inf;
    __shared__ KeyT skeys[kBigSmemKeys];
    __shared__ uint32_t item_s;
    __shared__ uint32_t sh_cnt[4];
    __shared__ unsigned long long sh_acc;
    const uint32_t tid = threadIdx.x;
    while (true) {
        if (tid == 0) item_s = atomicAdd(&ctr->big_cursor[chunk], 1u);
        __syncthreads();
        const uint32_t item = item_s;
        if (item >= ctr->big_count[chunk]) break;
        const uint32_t l = big_list[l0 + item];
        const uint32_t seg = seg_off[l], cap = seg_off[l + 1] - seg;
        if ((uint64_t)seg + cap > vals_cap) { __syncthreads(); continue; }     // see k_locus_median
        const unsigned long long cur = cursor[l];
        const uint32_t nf = min((uint32_t)cur, cap), nb = min((uint32_t)(cur >> 32), cap - nf);
        uint32_t ntot = nf + nb;
        const uint32_t n1 = unphased ? (ntot >> 1) : nf;
        const uint32_t n2 = ntot - n1;
        volatile KeyT *a;
        if (ntot <= (uint32_t)kBigSmemKeys) {
            for (uint32_t i = tid; i < ntot; i += blockDim.x) {
                KeyT v;
                if (i < nf) v = vals[seg + i];
                else v = vals[seg + cap - nb + (i - nf)] | (unphased ? (KeyT)0 : hap);
                skeys[i] = v;
            }
            a = skeys;
        } else {
            // sort the whole segment in place; the unused gap between front and back becomes +inf keys
            for (uint32_t i = nf + tid; i < cap; i += blockDim.x) {
                if (i < cap - nb) vals[seg + i] = inf;
                else if (!unphased) vals[seg + i] |= hap;
            }
            a = vals + seg;
            ntot = cap;
        }
        __syncthreads();
        // all-ascending bitonic network with virtual +inf padding (comparators touching i >= ntot are no-ops)
        uint32_t npow = 1;
        while (npow < ntot) npow <<= 1;
        for (uint32_t blk = 2; blk <= npow; blk <<= 1) {
            for (uint32_t i = tid; i < npow; i += blockDim.x) {
                const uint32_t j = i ^ (blk - 1);
                if (i < j && j < ntot) {
                    const KeyT x = a[i], y = a[j];
                    if (x > y) { a[i] = y; a[j] = x; }
                }
            }
            __syncthreads();
            for (uint32_t d = blk >> 2; d >= 1; d >>= 1) {
                for (uint32_t i = tid; i < npow; i += blockDim.x) {
                    const uint32_t j = i ^ d;
                    if (i < j && j < ntot) {
                        const KeyT x = a[i], y = a[j];
                        if (x > y) { a[i] = y; a[j] = x; }
                    }
                }
                __syncthreads();
            }
        }
        int64_t t1, t2;
        bool ok1, ok2, panicked = false;
        block_part_median(a, 0, n1, support, &t1, &ok1, &panicked, sh_cnt, &sh_acc);
        __syncthreads();
        block_part_median(a, n1, n2, support, &t2, &ok2, &panicked, sh_cnt, &sh_acc);
        if (tid == 0) {
            twice_h1[l] = t1;
            twice_h2[l] = t2;
            valid[l] = (uint8_t)((ok1 ? 1u : 0u) | (ok2 ? 2u : 0u));
            if (panicked) atomicOr(&ctr->flags, kFlagMedianEmpty);
        }
        __syncthreads();
    }
}

}  // namespace inq
