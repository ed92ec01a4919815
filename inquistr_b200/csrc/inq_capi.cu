// inq_capi.cu -- extern "C" boundary of libinqcall.so (see include/inqcall.h).
// Host-side orchestration only: device memory, H2D/D2H copies, kernel launches and timing.
// No CPU implementation of the hot path lives here: without a CUDA device every entry fails.
//
// One genotyping pass is a small DAG over four streams (DESIGN.md section 3b):
//   S0  counter memset, k_cigar_scan over the whole CIGAR stream, then the prefix sum over its warp-tile totals
//       (k_exclusive_scan2)
//   S1  k_zero, k_join_ranges + two offset scans (next to the CIGAR scan), then k_pair_eval once S0 is done
//   S2  k_locus_median (+ the CTA-path kernel where the last pass had deep loci) per catalog chunk; the counters go
//       home from here
//   S3  k_push_results: finished chunks stored into the caller's pinned arrays (copy engines when they are not mapped)
// The steady state (same reads, same parameters, same pinned outputs) is replayed from a CUDA graph; the first call
// of a shape and every retry (speculative buffer regrown, CTA-path guess wrong) launch the same DAG directly.
#include "../../include/inqcall.h"
#include "inq_device.cuh"
#include "host/catalog_reach.hpp"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace inq;

namespace {

thread_local std::string g_create_error;

template <typename T>
struct DevBuf {
    T *p = nullptr;
    uint64_t cap = 0;   // elements
};

// driver entry points (libcuda is not linked; they are fetched through the runtime)
typedef CUresult (*tmap_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*mem_reserve_fn)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long);
typedef CUresult (*mem_create_fn)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long);
typedef CUresult (*mem_map_fn)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
typedef CUresult (*mem_access_fn)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t);
typedef CUresult (*mem_unmap_fn)(CUdeviceptr, size_t);
typedef CUresult (*mem_release_fn)(CUmemGenericAllocationHandle);
typedef CUresult (*mem_free_fn)(CUdeviceptr, size_t);
typedef CUresult (*mem_gran_fn)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags);

struct DriverApi {
    tmap_encode_fn tmap_encode = nullptr;
    mem_reserve_fn reserve = nullptr;
    mem_create_fn create = nullptr;
    mem_map_fn map = nullptr;
    mem_access_fn set_access = nullptr;
    mem_unmap_fn unmap = nullptr;
    mem_release_fn release = nullptr;
    mem_free_fn addr_free = nullptr;
    mem_gran_fn granularity = nullptr;
    const char *missing = nullptr;    // the first of the entry points above that the driver does not provide
};

void *driver_symbol(const char *name, const char *&missing)
{
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) fn = nullptr;
    if (!fn && !missing) missing = name;
    return fn;
}

const DriverApi &driver()
{
    static DriverApi d = [] {
        DriverApi a;
        a.tmap_encode = (tmap_encode_fn)driver_symbol("cuTensorMapEncodeTiled", a.missing);
        a.reserve = (mem_reserve_fn)driver_symbol("cuMemAddressReserve", a.missing);
        a.create = (mem_create_fn)driver_symbol("cuMemCreate", a.missing);
        a.map = (mem_map_fn)driver_symbol("cuMemMap", a.missing);
        a.set_access = (mem_access_fn)driver_symbol("cuMemSetAccess", a.missing);
        a.unmap = (mem_unmap_fn)driver_symbol("cuMemUnmap", a.missing);
        a.release = (mem_release_fn)driver_symbol("cuMemRelease", a.missing);
        a.addr_free = (mem_free_fn)driver_symbol("cuMemAddressFree", a.missing);
        a.granularity = (mem_gran_fn)driver_symbol("cuMemGetAllocationGranularity", a.missing);
        return a;
    }();
    return d;
}

// The CIGAR unit stream (the one multi-GB buffer) lives in a reserved virtual address range that is
// backed by physical chunks as reads arrive: growing it neither copies the stream nor moves its base
// address (the TMA tensor map and a captured graph stay valid).
struct VmStream {
    CUdeviceptr base = 0;
    size_t reserved = 0, mapped = 0, gran = 0;
    std::vector<std::pair<CUmemGenericAllocationHandle, size_t>> chunks;
};

enum {
    EV_START = 0, EV_END, EV_INDEX, EV_JOIN, EV_MED0, EV_MED1, EV_D2H, EV_H2D0, EV_H2D1,
    EV_SCAN0, EV_SCAN1,                         // start / end of k_cigar_scan
    EV_PAIR0, EV_PAIR1,                         // start / end of k_pair_eval
    EV_COUNT
};
// dependency-only events (no timing)
enum {
    DEP_FORK = 0, DEP_JOIN_DONE, DEP_S1_DONE, DEP_S2_DONE, DEP_S3_DONE, DEP_ZEROED, DEP_SCAN_ONLY, DEP_SCANNED, DEP_PAIRED,
    DEP_CHUNK,                                  // + c: median chunk c done
    DEP_COUNT = DEP_CHUNK + kMaxMedianChunks
};

struct MedianChunk {
    uint32_t l0, l1;
};

// How the medians are cut up; rebuilt whenever the reads or the catalog change.
struct Plan {
    bool valid = false;
    uint64_t data_gen = 0;
    int n_chunks = 0;
    MedianChunk chunk[kMaxMedianChunks];
    bool reads_sorted = false;
    // the CTA-path median kernel of a chunk is only launched where the last completed pass over the same reads had
    // deep loci (it is empty almost everywhere and costs a launch on the S2 chain per chunk); verified after every
    // pass from the per-chunk counters, like the speculative buffer sizes
    bool big_known = false;
    bool need_big[kMaxMedianChunks] = {};
};

struct GraphKey {
    uint64_t data_gen = 0, buf_gen = 0;
    uint32_t minlen = 0, support = 0;
    int unphased = 0, timing = 0;
    const void *o1 = nullptr, *o2 = nullptr, *ov = nullptr;
    bool wide_keys = false;
    bool operator==(const GraphKey &o) const
    {
        return data_gen == o.data_gen && buf_gen == o.buf_gen && minlen == o.minlen && support == o.support &&
               unphased == o.unphased && timing == o.timing && o1 == o.o1 && o2 == o.o2 && ov == o.ov &&
               wide_keys == o.wide_keys;
    }
};

}  // namespace

struct inq_ctx {
    int device = 0;
    int sm_count = 0;
    int scan_ctas_per_sm = 1;
    cudaStream_t stream = nullptr;        // S0
    cudaStream_t stream_join = nullptr;   // S1: join, pair evaluation
    cudaStream_t stream_med = nullptr;    // S2: medians
    cudaStream_t stream_copy = nullptr;   // S3: result copies
    std::string err;

    // options (inq_set_option)
    int opt_graph = 1;
    int opt_timing = 1;

    // locus catalog
    int32_t n_contigs = 0;
    int64_t L = 0;
    DevBuf<int64_t> contig_off;
    DevBuf<int32_t> lstart, lend, lpmax;
    inqhost::CatalogReach reach;          // host index of the catalog (valid while L > 0): which reads inq_push_reads_routed takes
    void *h_route_stage = nullptr;        // pinned staging of inq_push_reads_routed when the kept reads are scattered

    // reads: C BAM words (the statistics count them), stored as U 16-bit units (inq_device.cuh, "CIGAR units")
    uint64_t R = 0, C = 0, U = 0;
    DevBuf<int32_t> contig, rs, re;
    DevBuf<uint8_t> mapq, hp, flags;
    DevBuf<uint64_t> cig_off, unit_off;
    VmStream vm;
    // encoding at push: a double-buffered staging ring of BAM words and the per-chunk unit counts / offsets
    DevBuf<uint32_t> push_stage, push_cnt, push_off;
    DevBuf<uint64_t> push_desc;
    DevBuf<unsigned int> push_ctr;        // tile counter and overflow flag of the offset scan
    cudaEvent_t push_landed[2] = {}, push_free[2] = {};
    uint32_t *d_unsorted = nullptr;       // != 0: the pushed reads are not sorted by (contig, ref_start)

    // work buffers
    DevBuf<uint32_t> cand_lo, cand_n, ev_off, delta, lcnt, seg_off, big_list;
    DevBuf<unsigned long long> cursor;
    DevBuf<uint32_t> wt_sbase, tile_first;
    DevBuf<uint2> rd_pre, wt, wtot;
    DevBuf<uint64_t> desc_scan, desc_wt;
    DevBuf<uint32_t> vals;                // call keys, one per candidate: 32-bit words, two per key with 64-bit keys
    DevBuf<uint2> evraw;
    CUtensorMap tmap;                 // 2-D view of the unit stream: rows of 32 words (64 units), 128B swizzle
    const void *tmap_base = nullptr;
    uint64_t tmap_rows = 0;
    DevBuf<uint2> events;
    DevBuf<int64_t> t1, t2;
    DevBuf<uint8_t> valid;
    DevCounters *d_ctr = nullptr;
    DevCounters *h_ctr = nullptr;     // pinned
    uint32_t *h_total = nullptr;      // pinned
    void *h_stage = nullptr;          // pinned staging of the results when the caller's arrays are pageable
    size_t h_stage_bytes = 0;

    cudaEvent_t ev[EV_COUNT] = {};
    cudaEvent_t dep[DEP_COUNT] = {};
    float ms_h2d = 0.f;
    uint64_t last_n_events = 0;

    uint64_t data_gen = 1, buf_gen = 1;
    uint64_t wide_gen = 0;                // == data_gen: these reads have a call outside 30 bits, the pass uses 64-bit keys
    Plan plan;
    cudaGraphExec_t graph = nullptr;
    GraphKey graph_key, last_key;
    bool have_last_key = false;
    uint32_t graph_launches = 0;
};

namespace {

int fail(inq_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

#define CU_TRY(ctx, call)                                                                      \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? INQ_ERR_NOMEM : INQ_ERR_CUDA,   \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

void drop_graph(inq_ctx *ctx)
{
    if (ctx->graph) cudaGraphExecDestroy(ctx->graph);
    ctx->graph = nullptr;
}

// grow-only device buffer; keeps the first `keep` elements
template <typename T>
int ensure(inq_ctx *ctx, DevBuf<T> &b, uint64_t need, uint64_t keep = 0, double growth = 1.0)
{
    if (need <= b.cap) return INQ_OK;
    uint64_t cap = std::max<uint64_t>(need, (uint64_t)(b.cap * growth));
    T *np = nullptr;
    CU_TRY(ctx, cudaMalloc(&np, std::max<uint64_t>(cap, 1) * sizeof(T)));
    if (keep && b.p) {
        cudaError_t e = cudaMemcpyAsync(np, b.p, std::min<uint64_t>(keep, b.cap) * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { cudaFree(np); return fail(ctx, INQ_ERR_CUDA, "device copy failed: %s", cudaGetErrorString(e)); }
    }
    if (b.p) cudaFree(b.p);
    b.p = np;
    b.cap = cap;
    ++ctx->buf_gen;                   // a captured graph holds the old pointer
    return INQ_OK;
}

// The call keys are 32 bits wide until a pass over the current reads meets a call outside [-2^29, 2^29) (the pair kernel
// raises kFlagWideCall); from then on, until the reads change, they are 64 bits wide.
bool wide_keys(const inq_ctx *ctx) { return ctx->wide_gen == ctx->data_gen; }
uint64_t vals_keys(const inq_ctx *ctx) { return wide_keys(ctx) ? ctx->vals.cap / 2 : ctx->vals.cap; }
int ensure_vals(inq_ctx *ctx, uint64_t keys) { return ensure(ctx, ctx->vals, wide_keys(ctx) ? 2 * keys : keys); }

template <typename T>
void release(DevBuf<T> &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

#define TRY(x) do { int rc_ = (x); if (rc_ != INQ_OK) return rc_; } while (0)

uint64_t round_up(uint64_t v, uint64_t m) { return (v + m - 1) / m * m; }

void vm_release(VmStream &vm)
{
    const DriverApi &d = driver();
    size_t off = 0;
    for (auto &c : vm.chunks) {
        d.unmap(vm.base + off, c.second);
        d.release(c.first);
        off += c.second;
    }
    vm.chunks.clear();
    if (vm.base) d.addr_free(vm.base, vm.reserved);
    vm = VmStream();
}

// make sure the first `bytes` of the stream are backed by device memory
int vm_ensure(inq_ctx *ctx, size_t bytes)
{
    VmStream &vm = ctx->vm;
    const DriverApi &d = driver();
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof(prop));
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = ctx->device;
    if (!vm.base) {
        if (d.granularity(&vm.gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || !vm.gran)
            return fail(ctx, INQ_ERR_CUDA, "cuMemGetAllocationGranularity failed");
        size_t total = 0, free_b = 0;
        CU_TRY(ctx, cudaMemGetInfo(&free_b, &total));
        vm.reserved = round_up(total, vm.gran);              // address space only: the whole device, nothing committed
        if (d.reserve(&vm.base, vm.reserved, 1u << 21, 0, 0) != CUDA_SUCCESS) { vm.base = 0; return fail(ctx, INQ_ERR_NOMEM, "cuMemAddressReserve(%zu) failed", vm.reserved); }
    }
    if (bytes <= vm.mapped) return INQ_OK;
    if (bytes > vm.reserved) return fail(ctx, INQ_ERR_NOMEM, "CIGAR stream of %zu bytes exceeds the device", bytes);
    // geometric chunk sizes keep the number of mappings small (64 MB .. 2 GB)
    size_t want = std::max<size_t>(bytes - vm.mapped, std::min<size_t>(std::max<size_t>(vm.mapped / 2, 64u << 20), 2048ull << 20));
    want = std::min(round_up(want, vm.gran), vm.reserved - vm.mapped);
    CUmemGenericAllocationHandle h;
    if (d.create(&h, want, &prop, 0) != CUDA_SUCCESS) {
        want = round_up(bytes - vm.mapped, vm.gran);         // no room for the slack: take exactly what is needed
        if (d.create(&h, want, &prop, 0) != CUDA_SUCCESS) return fail(ctx, INQ_ERR_NOMEM, "cuMemCreate(%zu) failed", want);
    }
    if (d.map(vm.base + vm.mapped, want, 0, h, 0) != CUDA_SUCCESS) { d.release(h); return fail(ctx, INQ_ERR_CUDA, "cuMemMap failed"); }
    CUmemAccessDesc acc;
    memset(&acc, 0, sizeof(acc));
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (d.set_access(vm.base + vm.mapped, want, &acc, 1) != CUDA_SUCCESS) {
        d.unmap(vm.base + vm.mapped, want);
        d.release(h);
        return fail(ctx, INQ_ERR_CUDA, "cuMemSetAccess failed");
    }
    vm.chunks.emplace_back(h, want);
    vm.mapped += want;
    return INQ_OK;
}

uint16_t *cigar_ptr(inq_ctx *ctx) { return reinterpret_cast<uint16_t *>(ctx->vm.base); }

// (re)build the TMA descriptor of the unit stream: uint32 [rows][32] (unit pairs), box = one 4 KB warp tile, 128B swizzle
int make_tensor_map(inq_ctx *ctx, uint64_t n_units_padded)
{
    const uint64_t rows = n_units_padded / 64;
    if (ctx->tmap_base == cigar_ptr(ctx) && ctx->tmap_rows == rows) return INQ_OK;
    const cuuint64_t gdim[2] = {32, rows};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {32, (cuuint32_t)(kWarpTileUnits / 64)};    // one warp tile
    const cuuint32_t estride[2] = {1, 1};
    CUresult r = driver().tmap_encode(&ctx->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, cigar_ptr(ctx), gdim, gstride, box, estride,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, INQ_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    ctx->tmap_base = cigar_ptr(ctx);
    ctx->tmap_rows = rows;
    ++ctx->buf_gen;                   // the tensor map is a kernel argument of a captured graph
    return INQ_OK;
}

// Room for nU units of the stream, padded to a tile boundary (+1 tile of slack). The stream grows in place; what
// must survive a regrow of tile_first are the entries of the `keep` units written so far: every warp tile up to
// their padded end plus the sentinel slot.
int reserve_units(inq_ctx *ctx, uint64_t nU, uint64_t keep)
{
    const uint64_t need_units = round_up(nU, kTileUnits) + kTileUnits;
    TRY(vm_ensure(ctx, need_units * sizeof(uint16_t)));
    TRY(ensure(ctx, ctx->tile_first, ctx->vm.mapped / 2 / kWarpTileUnits + 2, keep ? round_up(keep, kTileUnits) / kWarpTileUnits + 1 : 0, 1.0));
    return INQ_OK;
}

int reserve_reads(inq_ctx *ctx, uint64_t nR, uint64_t nU, double growth)
{
    const uint64_t R = ctx->R;
    TRY(ensure(ctx, ctx->contig, nR, R, growth));
    TRY(ensure(ctx, ctx->rs, nR, R, growth));
    TRY(ensure(ctx, ctx->re, nR, R, growth));
    TRY(ensure(ctx, ctx->mapq, nR, R, growth));
    TRY(ensure(ctx, ctx->hp, nR, R, growth));
    TRY(ensure(ctx, ctx->flags, nR, R, growth));
    TRY(ensure(ctx, ctx->cig_off, nR + 1, R + 1, growth));
    TRY(ensure(ctx, ctx->unit_off, nR + 1, R + 1, growth));
    return reserve_units(ctx, nU, R ? ctx->U : 0);
}

// ---- small kernels of the orchestration layer ---------------------------------------------------

// reads [r0, r0 + n) continue a (contig, ref_start)-sorted sequence? contig compares unsigned so that
// unmapped reads (tid -1) sort last, as in a coordinate-sorted BAM
__global__ void k_check_sorted(const int32_t *__restrict__ contig, const int32_t *__restrict__ rs, uint64_t r0, uint64_t n,
                               uint32_t *__restrict__ unsorted)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = r0 + i;
        if (r == 0) continue;
        const uint32_t ca = (uint32_t)contig[r - 1], cb = (uint32_t)contig[r];
        if (ca > cb || (ca == cb && rs[r - 1] > rs[r])) *unsorted = 1u;
    }
}

// everything a pass needs zeroed besides the counters, in one launch (six small memsets cost ~15 us of launch latency
// on the critical path of a small workload)
struct ZeroJob { void *p; uint64_t bytes; };
struct ZeroJobs { ZeroJob j[6]; int n; };
// The results of one median chunk go home through a kernel that stores into the caller's pinned (mapped) arrays:
// one launch in place of three copy-engine operations, whose ~10 us apiece of fixed latency is what a chunk's
// transfer costs at the per-rank sizes of a multi-GPU run. 16-byte streaming stores between the aligned edges
// of each array (source and destination share the index; when they do not share the alignment: bytes).
__device__ __forceinline__ void push_bytes(unsigned char *__restrict__ dst, const unsigned char *__restrict__ src, size_t n, uint32_t tid, uint32_t stride)
{
    if (((reinterpret_cast<uintptr_t>(dst) ^ reinterpret_cast<uintptr_t>(src)) & 15u) != 0) {
        if ((((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src) | n) & 7u) == 0)) {
            for (size_t i = tid; i < n / 8; i += stride) __stcs(reinterpret_cast<unsigned long long *>(dst) + i, reinterpret_cast<const unsigned long long *>(src)[i]);
        } else {
            for (size_t i = tid; i < n; i += stride) dst[i] = src[i];
        }
        return;
    }
    const size_t head = min(n, (size_t)((16u - (reinterpret_cast<uintptr_t>(src) & 15u)) & 15u));
    const size_t nv = (n - head) / 16, tail0 = head + nv * 16;
    if (tid < head) dst[tid] = src[tid];
    const uint4 *sv = reinterpret_cast<const uint4 *>(src + head);
    uint4 *dv = reinterpret_cast<uint4 *>(dst + head);
    for (size_t i = tid; i < nv; i += stride) __stcs(dv + i, sv[i]);
    if (tid < n - tail0) dst[tail0 + tid] = src[tail0 + tid];
}

constexpr unsigned kPushCtas = 8;     // the stores are PCIe-bound: a few SMs' worth is plenty

__global__ void __launch_bounds__(256)
k_push_results(uint32_t l0, uint32_t l1, const int64_t *__restrict__ t1, const int64_t *__restrict__ t2, const uint8_t *__restrict__ valid,
               int64_t *__restrict__ o1, int64_t *__restrict__ o2, uint8_t *__restrict__ ov)
{
    const uint32_t stride = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t n = l1 - l0;
    push_bytes(reinterpret_cast<unsigned char *>(o1 + l0), reinterpret_cast<const unsigned char *>(t1 + l0), n * 8, tid, stride);
    push_bytes(reinterpret_cast<unsigned char *>(o2 + l0), reinterpret_cast<const unsigned char *>(t2 + l0), n * 8, tid, stride);
    push_bytes(ov + l0, valid + l0, n, tid, stride);
}

__global__ void k_zero(ZeroJobs jobs)
{
    for (int k = 0; k < jobs.n; ++k) {
        uint4 *p = static_cast<uint4 *>(jobs.j[k].p);
        const uint64_t n16 = jobs.j[k].bytes / 16;
        for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
    }
}

struct RunParams {
    uint32_t minlen, support;
    int unphased;
    int64_t *o1, *o2;
    uint8_t *ov;
    int timing;                             // 0: none; 1: pass + CIGAR scan (3 event records); 2: every stage (~10, ~5 us apiece in a replayed graph)
    int64_t *d1 = nullptr, *d2 = nullptr;   // device views of o1/o2/ov (mapped pinned memory); null: use the copy engines
    uint8_t *dv = nullptr;
};

// The medians run in catalog chunks so that the transfer of one runs under the medians of the next; the very last
// chunk is small (its transfer is the exposed one). profiles/r2_sweep_median_pieces.jsonl: flat within 1 % around these.
constexpr int64_t kMedianPieces = 12;     // median chunks per pass
constexpr int64_t kMinPiece = 1 << 16;    // ... but no chunk smaller than this many loci (the last one: a quarter of it)

// Cut the catalog into median chunks and read whether the reads are sorted. Needs one small device read-back, so it is
// cached until the reads or the catalog change.
int build_plan(inq_ctx *ctx)
{
    Plan &pl = ctx->plan;
    if (pl.valid && pl.data_gen == ctx->data_gen) return INQ_OK;
    pl = Plan();
    const int64_t L = ctx->L;
    if (ctx->R && L) {
        cudaStream_t s = ctx->stream;
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total + 8, ctx->d_unsorted, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU_TRY(ctx, cudaStreamSynchronize(s));
        pl.reads_sorted = ctx->h_total[8] == 0;
    }
    const int64_t piece = std::max<int64_t>(kMinPiece, (L + kMedianPieces - 1) / kMedianPieces);
    const int64_t last_piece = std::max<int64_t>(kMinPiece / 4, L / (4 * kMedianPieces));
    for (int64_t a = 0; a < L;) {
        int64_t e = std::min(L, a + piece);
        if (L - a > 2 * last_piece && e > L - last_piece) e = L - last_piece;
        if (pl.n_chunks == kMaxMedianChunks - 1) e = L;
        pl.chunk[pl.n_chunks++] = MedianChunk{(uint32_t)a, (uint32_t)e};
        a = e;
    }
    pl.valid = true;
    pl.data_gen = ctx->data_gen;
    return INQ_OK;
}

uint32_t loc_scan_tiles(int64_t L) { return (uint32_t)(((uint64_t)L + 1 + kXsTile - 1) / kXsTile); }

// k_join_ranges, then the two offset scans over its difference array: lcnt[i+1] = number of candidate reads of locus
// i, seg_off = exclusive scan of those counts. delta, desc_scan and the counters must be zero.
int launch_join(inq_ctx *ctx, int unphased, cudaStream_t s)
{
    const int64_t L = ctx->L;
    const uint64_t R = ctx->R;
    const uint32_t tiles = loc_scan_tiles(L);
    ReadView rv{ctx->contig.p, ctx->rs.p, ctx->re.p, ctx->mapq.p, ctx->hp.p, ctx->flags.p, ctx->cig_off.p, R};
    LocusView lv{ctx->contig_off.p, ctx->lstart.p, ctx->lend.p, ctx->lpmax.p, ctx->n_contigs};
    k_join_ranges<<<(unsigned)((R + 255) / 256), 256, 0, s>>>(rv, lv, unphased, ctx->cand_lo.p, ctx->cand_n.p, ctx->delta.p, ctx->d_ctr);
    const unsigned g = std::min<unsigned>(tiles, (unsigned)ctx->sm_count * 4);
    k_exclusive_scan<<<g, kXsThreads, 0, s>>>(ctx->delta.p, ctx->lcnt.p, (uint64_t)L + 1, tiles, ctx->desc_scan.p,
                                              &ctx->d_ctr->scan_counter[2], nullptr);
    k_exclusive_scan<<<g, kXsThreads, 0, s>>>(ctx->lcnt.p + 1, ctx->seg_off.p, (uint64_t)L, tiles,
                                              ctx->desc_scan.p + tiles + 1, &ctx->d_ctr->scan_counter[3], &ctx->d_ctr->flags);
    CU_TRY(ctx, cudaGetLastError());
    return INQ_OK;
}

// Enqueue one whole pass on the four streams, starting and ending on S0. `capturing`: inside a stream
// capture (timing events are recorded as external event nodes).
int enqueue_pass(inq_ctx *ctx, const RunParams &rp, bool capturing, uint32_t *n_launches)
{
    const Plan &pl = ctx->plan;
    const int64_t L = ctx->L;
    const uint64_t R = ctx->R, U = ctx->U;
    cudaStream_t s0 = ctx->stream, s1 = ctx->stream_join, s2 = ctx->stream_med, s3 = ctx->stream_copy;
    const uint32_t ntiles = (uint32_t)((U + kTileUnits - 1) / kTileUnits);
    const uint64_t n_wt = (uint64_t)ntiles * (kTileUnits / kWarpTileUnits);
    const bool work = R && L;
    const bool scan = n_wt && L;
    uint32_t launches = 0;
    auto stamp = [&](int e, cudaStream_t s, int level = 2) -> cudaError_t {
        if (rp.timing < level) return cudaSuccess;
        return cudaEventRecordWithFlags(ctx->ev[e], s, capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
    };

    // S0 only needs the counters zeroed before the scan starts; everything the join / pair / median kernels need
    // zeroed is cleared on S1, off the scan's critical path
    CU_TRY(ctx, cudaMemsetAsync(ctx->d_ctr, 0, sizeof(DevCounters), s0));
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_FORK], s0));
    // (EV_START / EV_END are plain event records on S0 around the pass -- or around the graph launch --, made by
    // inq_genotype: no nodes of the graph)

    // ---- S1: K1 candidate ranges + difference array, then the per-locus segment offsets. Enqueued before the scan:
    //      the order decides whose CTAs the SMs see first.
    CU_TRY(ctx, cudaStreamWaitEvent(s1, ctx->dep[DEP_FORK], 0));
    {
        // (buffers come from cudaMalloc: 256-byte aligned; the sizes are rounded up to 16 bytes inside their capacity)
        ZeroJobs z;
        z.n = 0;
        auto add = [&](void *p, uint64_t bytes, uint64_t cap_bytes) { if (p && bytes) z.j[z.n++] = ZeroJob{p, std::min((bytes + 15) / 16 * 16, cap_bytes / 16 * 16)}; };
        uint64_t biggest = 0;
        if (L) {
            add(ctx->delta.p, ((uint64_t)L + 2) * sizeof(uint32_t), ctx->delta.cap * sizeof(uint32_t));
            add(ctx->seg_off.p, ((uint64_t)L + 2) * sizeof(uint32_t), ctx->seg_off.cap * sizeof(uint32_t));
            add(ctx->cursor.p, ((uint64_t)L + 1) * sizeof(unsigned long long), ctx->cursor.cap * sizeof(unsigned long long));
            add(ctx->desc_scan.p, 2 * ((uint64_t)loc_scan_tiles(L) + 1) * sizeof(uint64_t), ctx->desc_scan.cap * sizeof(uint64_t));
            biggest = ((uint64_t)L + 1) * sizeof(unsigned long long);
        }
        if (!ntiles) add(ctx->wt.p, 2 * sizeof(uint2), ctx->wt.cap * sizeof(uint2));      // no CIGAR units at all
        if (n_wt) add(ctx->desc_wt.p, ctx->desc_wt.cap * sizeof(uint64_t), ctx->desc_wt.cap * sizeof(uint64_t));
        if (z.n) {
            const unsigned g = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((std::max<uint64_t>(biggest, 4096) / 16 + 255) / 256, (uint64_t)ctx->sm_count * 4));
            k_zero<<<g, 256, 0, s1>>>(z);
            CU_TRY(ctx, cudaGetLastError());
        }
        CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_ZEROED], s1));
        CU_TRY(ctx, stamp(EV_INDEX, s1));
    }
    if (work) {
        TRY(launch_join(ctx, rp.unphased, s1));
        launches += 3;
        // the call buffer holds one slot per candidate; its size is only known on the device (checked after the pass)
        // (read home on S2, idle until the first medians: a copy-engine operation in front of k_pair_eval costs the chain ~10 us)
        CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_JOIN_DONE], s1));
        CU_TRY(ctx, cudaStreamWaitEvent(s2, ctx->dep[DEP_JOIN_DONE], 0));
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total, ctx->seg_off.p + L, sizeof(uint32_t), cudaMemcpyDeviceToHost, s2));
    }
    CU_TRY(ctx, stamp(EV_JOIN, s1));

    // ---- S0: K2, then the prefix sum over its warp-tile totals on the same stream, so that the join chain on S1
    //      (slow under the scan) has until the end of the scan; the scan's end is time-stamped on the idle S3
    CU_TRY(ctx, stamp(EV_SCAN0, s0));
    if (scan) {
        ScanParams sp;
        sp.tile_first = ctx->tile_first.p; sp.unit_off = ctx->unit_off.p; sp.units = cigar_ptr(ctx); sp.rd_pre = ctx->rd_pre.p;
        sp.wt = ctx->wtot.p; sp.wt_sbase = ctx->wt_sbase.p; sp.evraw = ctx->evraw.p; sp.ctr = ctx->d_ctr; sp.raw_cap = ctx->evraw.cap;
        sp.n_wt = n_wt; sp.ev_thr = scan_ev_thr(rp.minlen); sp.minlen = rp.minlen;
        // the unit field holds lengths up to 4094 exactly and 4095 for every longer I/D/S: from minlen 4095 on only
        // those long heads can be events, and k_cigar_scan<true> checks their full length
        const unsigned grid = (unsigned)std::min<uint64_t>((n_wt + kScanWarps - 1) / kScanWarps, (uint64_t)ctx->sm_count * ctx->scan_ctas_per_sm);
        if (rp.minlen >= kUnitLong) k_cigar_scan<true><<<grid, kCtaThreads, kScanSmemBytes, s0>>>(ctx->tmap, sp);
        else k_cigar_scan<false><<<grid, kCtaThreads, kScanSmemBytes, s0>>>(ctx->tmap, sp);
        ++launches;
        CU_TRY(ctx, cudaGetLastError());
    }
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_SCAN_ONLY], s0));
    if (rp.timing >= 1) {
        CU_TRY(ctx, cudaStreamWaitEvent(s3, ctx->dep[DEP_SCAN_ONLY], 0));
        CU_TRY(ctx, stamp(EV_SCAN1, s3, 1));
    }
    CU_TRY(ctx, cudaStreamWaitEvent(s0, ctx->dep[DEP_ZEROED], 0));       // desc_wt is cleared by k_zero
    if (scan) {
        const uint32_t xt = (uint32_t)((n_wt + kXsTile - 1) / kXsTile);
        const unsigned g = std::min<unsigned>(xt, (unsigned)ctx->sm_count * 4);
        uint64_t *dx = ctx->desc_wt.p, *dy = dx + xt + 1;
        k_exclusive_scan2<<<g, kXsThreads, 0, s0>>>(ctx->wtot.p, ctx->wt.p, n_wt, xt, dx, dy, &ctx->d_ctr->wt_scan_counter, &ctx->d_ctr->flags);
        ++launches;
        CU_TRY(ctx, cudaGetLastError());
    }
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_SCANNED], s0));

    // ---- S1: K2b once the stream is scanned ; S2: K3 per catalog chunk ; S3: result copies
    CU_TRY(ctx, cudaStreamWaitEvent(s1, ctx->dep[DEP_SCANNED], 0));
    CU_TRY(ctx, stamp(EV_PAIR0, s1));
    const bool wide = wide_keys(ctx);
    uint64_t *vals64 = reinterpret_cast<uint64_t *>(ctx->vals.p);
    const uint64_t vcap = vals_keys(ctx);
    if (work) {
        const unsigned threads = kPairWarps * 32;
        ReadView rv{ctx->contig.p, ctx->rs.p, ctx->re.p, ctx->mapq.p, ctx->hp.p, ctx->flags.p, ctx->cig_off.p, R};
        LocusView lv{ctx->contig_off.p, ctx->lstart.p, ctx->lend.p, ctx->lpmax.p, ctx->n_contigs};
        const EventSource es{ctx->unit_off.p, ctx->wt.p, ctx->rd_pre.p, ctx->wt_sbase.p, ctx->evraw.p, ctx->evraw.cap};
        const unsigned grid = (unsigned)((R + threads - 1) / threads);
        if (wide)
            k_pair_eval<uint64_t><<<grid, threads, sizeof(PairSmem), s1>>>(rv, 0, R, lv, rp.unphased, ctx->cand_lo.p, ctx->cand_n.p, es,
                                                                           ctx->seg_off.p, ctx->cursor.p, vals64, vcap, ctx->d_ctr);
        else
            k_pair_eval<uint32_t><<<grid, threads, sizeof(PairSmem), s1>>>(rv, 0, R, lv, rp.unphased, ctx->cand_lo.p, ctx->cand_n.p, es,
                                                                           ctx->seg_off.p, ctx->cursor.p, ctx->vals.p, vcap, ctx->d_ctr);
        ++launches;
        CU_TRY(ctx, cudaGetLastError());
    }
    CU_TRY(ctx, stamp(EV_PAIR1, s1));
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_PAIRED], s1));
    int64_t *o1 = rp.o1, *o2 = rp.o2;
    uint8_t *ov = rp.ov;
    for (int c = 0; c < pl.n_chunks; ++c) {
        const uint32_t l0 = pl.chunk[c].l0, l1 = pl.chunk[c].l1;
        if (c == 0) {
            // (S1 ran the join before the pair kernel: the first chunk also sees the empty segments of loci without reads)
            CU_TRY(ctx, cudaStreamWaitEvent(s2, ctx->dep[DEP_PAIRED], 0));
            CU_TRY(ctx, stamp(EV_MED0, s2));
        }
        const unsigned grid = (unsigned)(((uint64_t)(l1 - l0) * 32 + 255) / 256);
        if (wide)
            k_locus_median<uint64_t><<<grid, 256, 0, s2>>>(l0, l1, c, rp.unphased, rp.support, ctx->seg_off.p, ctx->cursor.p, vals64, vcap,
                                                           ctx->t1.p, ctx->t2.p, ctx->valid.p, ctx->big_list.p, ctx->d_ctr);
        else
            k_locus_median<uint32_t><<<grid, 256, 0, s2>>>(l0, l1, c, rp.unphased, rp.support, ctx->seg_off.p, ctx->cursor.p, ctx->vals.p, vcap,
                                                           ctx->t1.p, ctx->t2.p, ctx->valid.p, ctx->big_list.p, ctx->d_ctr);
        CU_TRY(ctx, cudaGetLastError());
        // the CTA path for the (rare) deep loci of the chunk, between two chunks on S2
        if (!pl.big_known || pl.need_big[c]) {
            const unsigned big_grid = (unsigned)ctx->sm_count * 2;
            if (wide)
                k_locus_median_big<uint64_t><<<big_grid, kBigThreads, 0, s2>>>(l0, c, rp.unphased, rp.support, ctx->seg_off.p, ctx->cursor.p, vals64, vcap,
                                                                               ctx->t1.p, ctx->t2.p, ctx->valid.p, ctx->big_list.p, ctx->d_ctr);
            else
                k_locus_median_big<uint32_t><<<big_grid, kBigThreads, 0, s2>>>(l0, c, rp.unphased, rp.support, ctx->seg_off.p, ctx->cursor.p, ctx->vals.p,
                                                                               vcap, ctx->t1.p, ctx->t2.p, ctx->valid.p, ctx->big_list.p, ctx->d_ctr);
            ++launches;
        }
        ++launches;
        CU_TRY(ctx, cudaGetLastError());
        CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_CHUNK + c], s2));
        CU_TRY(ctx, cudaStreamWaitEvent(s3, ctx->dep[DEP_CHUNK + c], 0));
        const size_t n = l1 - l0;
        if (rp.d1) {
            const unsigned g = (unsigned)std::min<size_t>(kPushCtas, (n + 2047) / 2048);
            k_push_results<<<std::max(g, 1u), 256, 0, s3>>>(l0, l1, ctx->t1.p, ctx->t2.p, ctx->valid.p, rp.d1, rp.d2, rp.dv);
            ++launches;
            CU_TRY(ctx, cudaGetLastError());
        } else {
            CU_TRY(ctx, cudaMemcpyAsync(o1 + l0, ctx->t1.p + l0, n * sizeof(int64_t), cudaMemcpyDeviceToHost, s3));
            CU_TRY(ctx, cudaMemcpyAsync(o2 + l0, ctx->t2.p + l0, n * sizeof(int64_t), cudaMemcpyDeviceToHost, s3));
            CU_TRY(ctx, cudaMemcpyAsync(ov + l0, ctx->valid.p + l0, n, cudaMemcpyDeviceToHost, s3));
        }
    }
    if (pl.n_chunks == 0) {                                   // nothing to do on S2/S3: keep them in the DAG for the join below
        CU_TRY(ctx, cudaStreamWaitEvent(s2, ctx->dep[DEP_FORK], 0));
        CU_TRY(ctx, stamp(EV_MED0, s2));
        CU_TRY(ctx, cudaStreamWaitEvent(s3, ctx->dep[DEP_FORK], 0));
    }
    CU_TRY(ctx, stamp(EV_MED1, s2));
    // total number of events = the last prefix
    if (scan) CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total + 2, ctx->wt.p + n_wt, sizeof(uint2), cudaMemcpyDeviceToHost, s1));
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_S1_DONE], s1));
    // the counters go home on S2 next to the last result copy (S3) instead of after it: S2 has seen every median kernel
    // (which raise flags), S1 every join / prefix / pair kernel, and those waited for the scans
    CU_TRY(ctx, cudaStreamWaitEvent(s2, ctx->dep[DEP_S1_DONE], 0));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, s2));
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_S2_DONE], s2));
    CU_TRY(ctx, stamp(EV_D2H, s3));
    CU_TRY(ctx, cudaEventRecord(ctx->dep[DEP_S3_DONE], s3));

    // ---- join everything on S0
    CU_TRY(ctx, cudaStreamWaitEvent(s0, ctx->dep[DEP_S1_DONE], 0));
    CU_TRY(ctx, cudaStreamWaitEvent(s0, ctx->dep[DEP_S2_DONE], 0));
    CU_TRY(ctx, cudaStreamWaitEvent(s0, ctx->dep[DEP_S3_DONE], 0));
    *n_launches = launches;
    return INQ_OK;
}

bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace

extern "C" {

const char *inq_version(void) { return "inquistr-b200 0.2.0 (sm_100a)"; }

const char *inq_last_error(const inq_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int inq_ctx_create(int device, inq_ctx **out)
{
    if (!out) return fail(nullptr, INQ_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, INQ_ERR_CUDA, "no CUDA device available (%s); libinqcall has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, INQ_ERR_ARG, "device %d out of range [0,%d)", device, n);
    inq_ctx *ctx = new inq_ctx();
    ctx->device = device;
    auto bail = [&](const char *what, cudaError_t err) {
        int rc = fail(nullptr, INQ_ERR_CUDA, "%s: %s", what, cudaGetErrorString(err));
        inq_ctx_destroy(ctx);
        return rc;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    if (prop.major < 10) {
        fail(nullptr, INQ_ERR_CUDA, "device %d is sm_%d%d; libinqcall is built for sm_100a only", device, prop.major, prop.minor);
        inq_ctx_destroy(ctx);
        return INQ_ERR_CUDA;
    }
    // the CIGAR stream lives in a virtual address range (cuMem*) and is read through a TMA tensor map
    if (const char *missing = driver().missing) {
        fail(nullptr, INQ_ERR_CUDA, "the CUDA driver does not provide %s, which libinqcall needs", missing);
        inq_ctx_destroy(ctx);
        return INQ_ERR_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    // the HBM-bound scan gets the SMs first; pair / median CTAs fill what its one CTA per SM leaves free. The result
    // pushes on S3 get them first too: they are PCIe-bound, and a push that waits behind the next median chunk's CTAs
    // leaves the link idle, so the last pushes would end the pass well after the last median
    int prio_lo = 0, prio_hi = 0;
    if ((e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi)) != cudaSuccess) return bail("cudaDeviceGetStreamPriorityRange", e);
    cudaStream_t *streams[4] = {&ctx->stream, &ctx->stream_join, &ctx->stream_med, &ctx->stream_copy};
    for (int i = 0; i < 4; ++i)
        if ((e = cudaStreamCreateWithPriority(streams[i], cudaStreamNonBlocking, (i == 0 || i == 3) ? prio_hi : prio_lo)) != cudaSuccess)
            return bail("cudaStreamCreate", e);
    for (int i = 0; i < EV_COUNT; ++i)
        if ((e = cudaEventCreate(&ctx->ev[i])) != cudaSuccess) return bail("cudaEventCreate", e);
    for (int i = 0; i < DEP_COUNT; ++i)
        if ((e = cudaEventCreateWithFlags(&ctx->dep[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (int i = 0; i < 2; ++i)
        if ((e = cudaEventCreateWithFlags(&ctx->push_landed[i], cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&ctx->push_free[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaMalloc(&ctx->d_ctr, sizeof(DevCounters))) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&ctx->d_unsorted, sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMemset(ctx->d_unsorted, 0, sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset", e);
    if ((e = cudaMallocHost(&ctx->h_ctr, sizeof(DevCounters))) != cudaSuccess) return bail("cudaMallocHost", e);
    if ((e = cudaMallocHost(&ctx->h_total, 64)) != cudaSuccess) return bail("cudaMallocHost", e);
    memset(ctx->h_ctr, 0, sizeof(DevCounters));
    if ((e = cudaFuncSetAttribute(k_cigar_scan<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScanSmemBytes)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_cigar_scan<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScanSmemBytes)) != cudaSuccess)
        return bail("cudaFuncSetAttribute(k_cigar_scan)", e);
    if ((e = cudaFuncSetAttribute(k_pair_eval<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem))) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_pair_eval<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PairSmem))) != cudaSuccess)
        return bail("cudaFuncSetAttribute(k_pair_eval)", e);
    int occ = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_cigar_scan<false>, kCtaThreads, kScanSmemBytes)) != cudaSuccess)
        return bail("occupancy(k_cigar_scan)", e);
    ctx->scan_ctas_per_sm = std::max(1, occ);
    *out = ctx;
    return INQ_OK;
}

void inq_ctx_destroy(inq_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    drop_graph(ctx);
    release(ctx->contig_off); release(ctx->lstart); release(ctx->lend); release(ctx->lpmax);
    release(ctx->contig); release(ctx->rs); release(ctx->re);
    release(ctx->mapq); release(ctx->hp); release(ctx->flags);
    release(ctx->cig_off); release(ctx->unit_off);
    release(ctx->push_stage); release(ctx->push_cnt); release(ctx->push_off); release(ctx->push_desc); release(ctx->push_ctr);
    if (ctx->vm.base) vm_release(ctx->vm);
    release(ctx->cand_lo); release(ctx->cand_n); release(ctx->ev_off);
    release(ctx->rd_pre); release(ctx->wt); release(ctx->wtot); release(ctx->wt_sbase); release(ctx->tile_first);
    release(ctx->desc_wt); release(ctx->evraw);
    release(ctx->delta); release(ctx->lcnt); release(ctx->seg_off); release(ctx->cursor); release(ctx->big_list);
    release(ctx->desc_scan); release(ctx->vals);
    release(ctx->events); release(ctx->t1); release(ctx->t2); release(ctx->valid);
    if (ctx->d_ctr) cudaFree(ctx->d_ctr);
    if (ctx->d_unsorted) cudaFree(ctx->d_unsorted);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    if (ctx->h_total) cudaFreeHost(ctx->h_total);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    if (ctx->h_route_stage) cudaFreeHost(ctx->h_route_stage);
    for (int i = 0; i < EV_COUNT; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < DEP_COUNT; ++i)
        if (ctx->dep[i]) cudaEventDestroy(ctx->dep[i]);
    for (int i = 0; i < 2; ++i) {
        if (ctx->push_landed[i]) cudaEventDestroy(ctx->push_landed[i]);
        if (ctx->push_free[i]) cudaEventDestroy(ctx->push_free[i]);
    }
    cudaStream_t streams[4] = {ctx->stream_copy, ctx->stream_med, ctx->stream_join, ctx->stream};
    for (auto s : streams)
        if (s) cudaStreamDestroy(s);
    delete ctx;
}

int inq_set_option(inq_ctx *ctx, const char *name, int64_t value)
{
    if (!ctx || !name) return INQ_ERR_ARG;
    const std::string n(name);
    if (n == "graph") ctx->opt_graph = value != 0;
    else if (n == "timing") {
        if (value < 0 || value > 2) return fail(ctx, INQ_ERR_ARG, "timing must be 0 (off), 1 (pass and CIGAR scan) or 2 (every stage)");
        ctx->opt_timing = (int)value;
    }
    else return fail(ctx, INQ_ERR_ARG, "unknown option '%s'", name);
    drop_graph(ctx);
    ctx->have_last_key = false;
    return INQ_OK;
}

int inq_host_alloc(size_t bytes, void **out)
{
    if (!out) return INQ_ERR_ARG;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return e == cudaErrorMemoryAllocation ? INQ_ERR_NOMEM : INQ_ERR_CUDA; }
    return INQ_OK;
}

int inq_host_free(void *p)
{
    if (!p) return INQ_OK;
    return cudaFreeHost(p) == cudaSuccess ? INQ_OK : INQ_ERR_CUDA;
}

int inq_set_loci(inq_ctx *ctx, int32_t n_contigs, const int64_t *contig_locus_offsets, const int32_t *start,
                 const int32_t *end)
{
    if (!ctx) return INQ_ERR_ARG;
    if (n_contigs < 0 || !contig_locus_offsets) return fail(ctx, INQ_ERR_ARG, "inq_set_loci: bad contig table");
    const int64_t L = contig_locus_offsets[n_contigs];
    if (contig_locus_offsets[0] != 0 || L < 0) return fail(ctx, INQ_ERR_ARG, "inq_set_loci: offsets must start at 0");
    for (int32_t c = 0; c < n_contigs; ++c)
        if (contig_locus_offsets[c + 1] < contig_locus_offsets[c]) return fail(ctx, INQ_ERR_ARG, "inq_set_loci: offsets not monotonic");
    if (L > 0 && (!start || !end)) return fail(ctx, INQ_ERR_ARG, "inq_set_loci: start/end are NULL");
    if ((uint64_t)L * 2 + 2 > 0x7FFFFFFFull) return fail(ctx, INQ_ERR_TOO_LARGE, "inq_set_loci: too many loci (%lld)", (long long)L);
    ctx->n_contigs = 0;
    ctx->L = 0;
    ++ctx->data_gen;
    // one host pass checks the catalog and builds the running max of `end` that the join reads (lpmax)
    const inqhost::CatalogFault bad = inqhost::catalog_fault(ctx->reach.build(n_contigs, contig_locus_offsets, start, end, 0, L));
    if (bad.code != INQ_OK) return fail(ctx, bad.code, "%s", bad.message);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    TRY(ensure(ctx, ctx->contig_off, (uint64_t)n_contigs + 1));
    TRY(ensure(ctx, ctx->lstart, (uint64_t)L));
    TRY(ensure(ctx, ctx->lend, (uint64_t)L));
    TRY(ensure(ctx, ctx->lpmax, (uint64_t)L));
    TRY(ensure(ctx, ctx->delta, (uint64_t)L + 2 + 4));            // (+ slack: k_zero clears in 16-byte units)
    TRY(ensure(ctx, ctx->lcnt, (uint64_t)L + 3));
    TRY(ensure(ctx, ctx->seg_off, (uint64_t)L + 2 + 4));
    TRY(ensure(ctx, ctx->cursor, (uint64_t)L + 1 + 2));
    TRY(ensure(ctx, ctx->big_list, (uint64_t)L + 1));
    TRY(ensure(ctx, ctx->desc_scan, 2 * (((uint64_t)L + 2 + kXsTile - 1) / kXsTile + 1) + 2));
    TRY(ensure(ctx, ctx->t1, (uint64_t)L));
    TRY(ensure(ctx, ctx->t2, (uint64_t)L));
    TRY(ensure(ctx, ctx->valid, (uint64_t)L));
    cudaStream_t s = ctx->stream;
    CU_TRY(ctx, cudaMemcpyAsync(ctx->contig_off.p, contig_locus_offsets, ((size_t)n_contigs + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (L) {
        CU_TRY(ctx, cudaMemcpyAsync(ctx->lstart.p, start, (size_t)L * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        CU_TRY(ctx, cudaMemcpyAsync(ctx->lend.p, end, (size_t)L * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        CU_TRY(ctx, cudaMemcpyAsync(ctx->lpmax.p, ctx->reach.pmax(), (size_t)L * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    }
    CU_TRY(ctx, cudaStreamSynchronize(s));
    ctx->n_contigs = n_contigs;
    ctx->L = L;
    return INQ_OK;
}

int inq_reserve_reads(inq_ctx *ctx, uint64_t n_reads, uint64_t n_cigar_words)
{
    if (!ctx) return INQ_ERR_ARG;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    // room for as many units as words: longer ops grow the stream in place when they are pushed
    return reserve_reads(ctx, std::max(n_reads, ctx->R), std::max(n_cigar_words, ctx->U), 1.0);
}

int inq_clear_reads(inq_ctx *ctx)
{
    if (!ctx) return INQ_ERR_ARG;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    ctx->R = 0;
    ctx->C = 0;
    ctx->U = 0;
    ++ctx->data_gen;
    CU_TRY(ctx, cudaMemsetAsync(ctx->d_unsorted, 0, sizeof(uint32_t), ctx->stream));
    return INQ_OK;
}

constexpr uint64_t kPushChunkWords = 1ull << 24;      // BAM words per encoding chunk (64 MB; a ring of up to two staging buffers)

unsigned grid_for(uint64_t n) { return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, 4096)); }

// Appends n reads whose CIGAR words are words[cigar_off[0] .. cigar_off[n]) (cigar_off need not start at 0).
// The words go to the device in chunks through a two-buffer staging ring on S3, so that the copy of chunk k+1
// overlaps the encoding of chunk k into units on S0: count the units of every word, scan the counts, read the
// chunk's total back (the stream may have to grow), write the units and the unit offsets of the reads that start
// in the chunk. The copies are asynchronous; the caller synchronises ctx->stream before the host arrays may change.
static int push_impl(inq_ctx *ctx, uint64_t n, const int32_t *contig, const int32_t *ref_start, const int32_t *ref_end,
                     const uint8_t *mapq, const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off, const uint32_t *words)
{
    const uint64_t w0 = cigar_off[0], nw = cigar_off[n] - w0;
    if (ctx->R + n >= 0xFFFFFFFFull) return fail(ctx, INQ_ERR_TOO_LARGE, "inq_push_reads: more than 2^32-2 reads");
    TRY(reserve_reads(ctx, ctx->R + n, ctx->U + nw, 1.5));
    const uint64_t stage_words = std::min(nw, kPushChunkWords);
    const uint64_t n_chunks = nw ? (nw + stage_words - 1) / stage_words : 0;
    const uint32_t max_xt = (uint32_t)((stage_words + kXsTile - 1) / kXsTile);
    if (nw) {
        // the second buffer of the ring only when there is a second chunk: a push of up to 64 MB of words holds one
        TRY(ensure(ctx, ctx->push_stage, std::min<uint64_t>(n_chunks, 2) * stage_words));
        TRY(ensure(ctx, ctx->push_cnt, stage_words));
        TRY(ensure(ctx, ctx->push_off, stage_words + 1));
        TRY(ensure(ctx, ctx->push_desc, (uint64_t)max_xt + 1));
        TRY(ensure(ctx, ctx->push_ctr, 2));
    }
    ++ctx->data_gen;
    cudaStream_t s = ctx->stream, sc = ctx->stream_copy;
    const uint64_t R0 = ctx->R, C0 = ctx->C, U0 = ctx->U;
    CU_TRY(ctx, cudaMemcpyAsync(ctx->contig.p + R0, contig, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->rs.p + R0, ref_start, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->re.p + R0, ref_end, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->mapq.p + R0, mapq, n, cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->hp.p + R0, hp, n, cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->flags.p + R0, flags, n, cudaMemcpyHostToDevice, s));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->cig_off.p + R0, cigar_off, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (C0 != w0) {                                              // batch-local offsets -> offsets into the device stream (mod 2^64)
        k_rebase_offsets<<<(unsigned)std::min<uint64_t>((n + 1 + 255) / 256, 8192), 256, 0, s>>>(ctx->cig_off.p + R0, n + 1, C0 - w0);
        CU_TRY(ctx, cudaGetLastError());
    }
    k_check_sorted<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 4096), 256, 0, s>>>(ctx->contig.p, ctx->rs.p, R0, n, ctx->d_unsorted);
    CU_TRY(ctx, cudaGetLastError());

    auto copy_chunk = [&](uint64_t k) -> int {
        const uint64_t a = k * stage_words, m = std::min(stage_words, nw - a);
        CU_TRY(ctx, cudaStreamWaitEvent(sc, ctx->push_free[k & 1], 0));      // the encoding of chunk k-2 is done with the buffer
        CU_TRY(ctx, cudaMemcpyAsync(ctx->push_stage.p + (k & 1) * stage_words, words + w0 + a, m * sizeof(uint32_t), cudaMemcpyHostToDevice, sc));
        CU_TRY(ctx, cudaEventRecord(ctx->push_landed[k & 1], sc));
        return INQ_OK;
    };
    uint64_t U1 = U0;
    if (n_chunks) TRY(copy_chunk(0));
    for (uint64_t k = 0; k < n_chunks; ++k) {
        if (k + 1 < n_chunks) TRY(copy_chunk(k + 1));
        const uint64_t a = k * stage_words, m = std::min(stage_words, nw - a);
        const uint32_t *src = ctx->push_stage.p + (k & 1) * stage_words;
        const uint32_t xt = (uint32_t)((m + kXsTile - 1) / kXsTile);
        CU_TRY(ctx, cudaStreamWaitEvent(s, ctx->push_landed[k & 1], 0));
        k_unit_count<<<grid_for(m), 256, 0, s>>>(src, m, ctx->push_cnt.p);
        CU_TRY(ctx, cudaMemsetAsync(ctx->push_desc.p, 0, ((uint64_t)xt + 1) * sizeof(uint64_t), s));
        CU_TRY(ctx, cudaMemsetAsync(ctx->push_ctr.p, 0, 2 * sizeof(unsigned int), s));
        k_exclusive_scan<<<std::min<unsigned>(xt, (unsigned)ctx->sm_count * 4), kXsThreads, 0, s>>>(
            ctx->push_cnt.p, ctx->push_off.p, m, xt, ctx->push_desc.p, ctx->push_ctr.p, ctx->push_ctr.p + 1);
        CU_TRY(ctx, cudaGetLastError());
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total + 12, ctx->push_off.p + m, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total + 13, ctx->push_ctr.p + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU_TRY(ctx, cudaStreamSynchronize(s));
        if (ctx->h_total[13]) return fail(ctx, INQ_ERR_TOO_LARGE, "inq_push_reads: %llu CIGAR words expand to 2^32 units or more", (unsigned long long)m);
        const uint64_t mu = ctx->h_total[12];
        TRY(reserve_units(ctx, U1 + mu, U1));
        k_unit_write<<<grid_for(m), 256, 0, s>>>(src, m, ctx->push_off.p, cigar_ptr(ctx) + U1);
        CU_TRY(ctx, cudaEventRecord(ctx->push_free[k & 1], s));
        // unit offsets of the reads that start in the chunk (the last chunk also takes those that start at its end)
        const uint64_t b = k + 1 == n_chunks ? nw + 1 : a + m;
        const uint64_t ra = (uint64_t)(std::lower_bound(cigar_off, cigar_off + n + 1, w0 + a) - cigar_off);
        const uint64_t rb = (uint64_t)(std::lower_bound(cigar_off, cigar_off + n + 1, w0 + b) - cigar_off);
        if (rb > ra) k_read_units<<<grid_for(rb - ra), 256, 0, s>>>(ctx->cig_off.p, R0 + ra, rb - ra, C0 + a, ctx->push_off.p, U1, ctx->unit_off.p);
        CU_TRY(ctx, cudaGetLastError());
        U1 += mu;
    }
    if (!nw) {
        k_read_units<<<grid_for(n + 1), 256, 0, s>>>(ctx->cig_off.p, R0, n + 1, 0, nullptr, U0, ctx->unit_off.p);
        CU_TRY(ctx, cudaGetLastError());
    }
    uint16_t *units = cigar_ptr(ctx);
    const uint64_t Upad = round_up(U1, kTileUnits);
    if (Upad > U1) CU_TRY(ctx, cudaMemsetAsync(units + U1, 0, (Upad - U1) * sizeof(uint16_t), s));
    {
        // reads starting per warp tile, for the tiles that gained units (k_cigar_scan leaves the tile-local
        // prefix of every read start in rd_pre); unit_off[R0 + n] is the sentinel and counts as a start
        const uint64_t t0 = U0 / kWarpTileUnits, t1 = Upad / kWarpTileUnits;
        k_tile_first<<<(unsigned)((t1 - t0 + 1 + 255) / 256), 256, 0, s>>>(ctx->unit_off.p, R0 + n + 1, t0, t1, ctx->tile_first.p);
        CU_TRY(ctx, cudaGetLastError());
    }
    ctx->R = R0 + n;
    ctx->C = C0 + nw;
    ctx->U = U1;
    return INQ_OK;
}

static int check_push_args(inq_ctx *ctx, uint64_t n, const int32_t *contig, const int32_t *ref_start, const int32_t *ref_end,
                           const uint8_t *mapq, const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off, const uint32_t *cigar_words)
{
    if (!contig || !ref_start || !ref_end || !mapq || !hp || !flags || !cigar_off) return fail(ctx, INQ_ERR_ARG, "inq_push_reads: NULL array");
    if (cigar_off[0] != 0) return fail(ctx, INQ_ERR_ARG, "inq_push_reads: cigar_off[0] must be 0");
    if (cigar_off[n] && !cigar_words) return fail(ctx, INQ_ERR_ARG, "inq_push_reads: cigar_words is NULL");
    return INQ_OK;
}

int inq_push_reads(inq_ctx *ctx, uint64_t n, const int32_t *contig, const int32_t *ref_start, const int32_t *ref_end,
                   const uint8_t *mapq, const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off,
                   const uint32_t *cigar_words)
{
    if (!ctx) return INQ_ERR_ARG;
    if (n == 0) return INQ_OK;
    TRY(check_push_args(ctx, n, contig, ref_start, ref_end, mapq, hp, flags, cigar_off, cigar_words));
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const bool first = ctx->R == 0;
    CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_H2D0], s));
    TRY(push_impl(ctx, n, contig, ref_start, ref_end, mapq, hp, flags, cigar_off, cigar_words));
    CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_H2D1], s));
    CU_TRY(ctx, cudaStreamSynchronize(s));       // host arrays may be reused by the caller after return
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[EV_H2D0], ctx->ev[EV_H2D1]);
    ctx->ms_h2d = (first ? 0.f : ctx->ms_h2d) + ms;
    return INQ_OK;
}

// Push only the reads of a batch that can matter to THIS context's catalog (see include/inqcall.h). With N contexts
// holding N contiguous catalog shards, handing every batch to every context routes the reads (reads at a cut go to
// both sides) without the caller knowing the cuts -- the host-side half of SURVEY 8e.
int inq_push_reads_routed(inq_ctx *ctx, uint64_t n, const int32_t *contig, const int32_t *ref_start, const int32_t *ref_end,
                          const uint8_t *mapq, const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off,
                          const uint32_t *cigar_words, uint32_t filter, int host_threads, uint64_t *n_taken)
{
    if (!ctx) return INQ_ERR_ARG;
    if (n_taken) *n_taken = 0;
    if (n == 0) return INQ_OK;
    TRY(check_push_args(ctx, n, contig, ref_start, ref_end, mapq, hp, flags, cigar_off, cigar_words));
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (!ctx->L) return INQ_OK;           // no catalog (or one without loci): no read reaches a locus
    const int nt = std::max(1, std::min(host_threads > 0 ? host_threads : (int)std::thread::hardware_concurrency(), 256));
    // 1. which reads would htslib's fetch return for some locus of this catalog (pos < end+10 && endpos > start-10,
    //    call.rs:285-288), minus the ones the per-read half of the filters rejects everywhere (call.rs:297-300,350-352)
    std::vector<uint8_t> keep(n);
    const inqhost::CatalogReach &reach = ctx->reach;
    auto mark = [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b; ++i)
            keep[i] = !((filter & INQ_ROUTE_DROP_LOW_MAPQ) && mapq[i] <= 10) && !((filter & INQ_ROUTE_DROP_NO_HP) && hp[i] == INQ_HP_ABSENT) &&
                      reach.reaches(contig[i], ref_start[i], ref_end[i]);
    };
    auto parallel = [&](uint64_t total, auto fn) {
        const uint64_t per = (total + nt - 1) / nt;
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t)
            if ((uint64_t)t * per < total) th.emplace_back([&, t] { fn((uint64_t)t * per, std::min(total, (uint64_t)(t + 1) * per)); });
        fn(0, std::min(total, per));
        for (auto &x : th) x.join();
    };
    parallel(n, mark);
    // 2. runs of kept reads. Short gaps are bridged (a read that reaches nothing is harmless on the device: the join
    //    gives it no candidates, and shipping it is cheaper than gathering around it): coordinate-sorted input and a
    //    contiguous catalog range give one run per contig
    constexpr uint64_t kBridge = 256;
    std::vector<std::pair<uint64_t, uint64_t>> runs;
    uint64_t taken = 0;
    for (uint64_t i = 0; i < n;) {
        if (!keep[i]) { ++i; continue; }
        uint64_t j = i + 1;
        while (j < n && keep[j]) ++j;
        if (!runs.empty() && i - runs.back().second <= kBridge) runs.back().second = j;
        else runs.emplace_back(i, j);
        i = j;
    }
    for (const auto &r : runs) taken += r.second - r.first;
    if (n_taken) *n_taken = taken;
    if (!taken) return INQ_OK;
    cudaStream_t s = ctx->stream;
    const bool first = ctx->R == 0;
    CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_H2D0], s));
    if (runs.size() <= 1024) {
        // coordinate-sorted input and a contiguous catalog range: a handful of runs, copied straight from the caller's arrays
        for (const auto &r : runs)
            TRY(push_impl(ctx, r.second - r.first, contig + r.first, ref_start + r.first, ref_end + r.first, mapq + r.first, hp + r.first,
                          flags + r.first, cigar_off + r.first, cigar_words));
    } else {
        // scattered: gather into pinned staging chunks (all host threads), one push per chunk
        constexpr uint64_t kStageWords = 16u << 20, kStageReads = 1u << 20;
        const size_t meta_bytes = kStageReads * 12 + (kStageReads + 1) * 8 + kStageReads * 3;
        if (!ctx->h_route_stage) CU_TRY(ctx, cudaMallocHost(&ctx->h_route_stage, kStageWords * 4 + meta_bytes + 64));
        uint32_t *sw = static_cast<uint32_t *>(ctx->h_route_stage);
        uint8_t *m = reinterpret_cast<uint8_t *>(sw + kStageWords);
        uint64_t *so = reinterpret_cast<uint64_t *>(m); m += (kStageReads + 1) * 8;
        int32_t *sc = reinterpret_cast<int32_t *>(m); m += kStageReads * 4;
        int32_t *ss = reinterpret_cast<int32_t *>(m); m += kStageReads * 4;
        int32_t *se = reinterpret_cast<int32_t *>(m); m += kStageReads * 4;
        uint8_t *sq = m; m += kStageReads;
        uint8_t *sh = m; m += kStageReads;
        uint8_t *sf = m;
        std::vector<uint64_t> idx;
        idx.reserve(kStageReads);
        size_t ri = 0;
        uint64_t pos_in_run = 0;
        while (ri < runs.size()) {
            idx.clear();
            uint64_t words = 0;
            so[0] = 0;
            while (ri < runs.size() && idx.size() < kStageReads) {
                const uint64_t i = runs[ri].first + pos_in_run;
                const uint64_t nw = cigar_off[i + 1] - cigar_off[i];
                if (nw > kStageWords) return fail(ctx, INQ_ERR_TOO_LARGE, "inq_push_reads_routed: a read has more CIGAR words than the staging buffer");
                if (words + nw > kStageWords) break;
                so[idx.size() + 1] = words + nw;
                idx.push_back(i);
                words += nw;
                if (++pos_in_run == runs[ri].second - runs[ri].first) { ++ri; pos_in_run = 0; }
            }
            const uint64_t cnt = idx.size();
            parallel(cnt, [&](uint64_t a, uint64_t b) {
                for (uint64_t k = a; k < b; ++k) {
                    const uint64_t i = idx[k];
                    sc[k] = contig[i]; ss[k] = ref_start[i]; se[k] = ref_end[i];
                    sq[k] = mapq[i]; sh[k] = hp[i]; sf[k] = flags[i];
                    memcpy(sw + so[k], cigar_words + cigar_off[i], (size_t)(cigar_off[i + 1] - cigar_off[i]) * 4);
                }
            });
            TRY(push_impl(ctx, cnt, sc, ss, se, sq, sh, sf, so, sw));
            CU_TRY(ctx, cudaStreamSynchronize(s));               // the staging buffer is refilled next
        }
    }
    CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_H2D1], s));
    CU_TRY(ctx, cudaStreamSynchronize(s));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[EV_H2D0], ctx->ev[EV_H2D1]);
    ctx->ms_h2d = (first ? 0.f : ctx->ms_h2d) + ms;
    return INQ_OK;
}

int inq_genotype(inq_ctx *ctx, uint32_t minlen, uint32_t support, int unphased, int64_t *twice_h1, int64_t *twice_h2,
                 uint8_t *valid_mask, inq_stats *stats)
{
    if (!ctx) return INQ_ERR_ARG;
    const int64_t L = ctx->L;
    const uint64_t R = ctx->R, C = ctx->C;
    if (L > 0 && (!twice_h1 || !twice_h2 || !valid_mask)) return fail(ctx, INQ_ERR_ARG, "inq_genotype: NULL output array");
    if (minlen >= (1u << 28)) minlen = (1u << 28) - 1;       // BAM op lengths have 28 bits: nothing is longer
    unphased = unphased != 0;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const uint64_t U = ctx->U;
    const uint32_t ntiles = (uint32_t)((U + kTileUnits - 1) / kTileUnits);
    if ((U + kTileUnits - 1) / kTileUnits > 0x7FFFFFFFull) return fail(ctx, INQ_ERR_TOO_LARGE, "too many CIGAR units");
    const uint64_t n_wt = (uint64_t)ntiles * (kTileUnits / kWarpTileUnits);
    const bool work = R && L;
    TRY(ensure(ctx, ctx->cand_lo, R));
    TRY(ensure(ctx, ctx->cand_n, R));
    TRY(ensure(ctx, ctx->rd_pre, R + 1));
    TRY(ensure(ctx, ctx->wt, n_wt + 2));
    TRY(ensure(ctx, ctx->wtot, n_wt + 2));
    TRY(ensure(ctx, ctx->wt_sbase, n_wt + 1));
    TRY(ensure(ctx, ctx->desc_wt, 2 * ((n_wt + kXsTile - 1) / kXsTile + 1)));       // even: k_zero clears it in 16-byte units
    if (ntiles) TRY(make_tensor_map(ctx, (uint64_t)ntiles * kTileUnits));
    const uint64_t raw_slack = (uint64_t)ctx->sm_count * ctx->scan_ctas_per_sm * kScanWarps * kEvChunk;
    // event storage is sized speculatively (1/16 of the words; checked and regrown after the run); it hands out
    // kEvChunk-slot chunks and a warp strands the remainder of its chunk whenever a tile does not fit any more
    if (ctx->evraw.cap == 0) TRY(ensure(ctx, ctx->evraw, C / 16 + 4096 + raw_slack));
    TRY(build_plan(ctx));

    // results go straight to the caller's arrays when those are pinned, otherwise through a pinned staging buffer
    const bool direct_out = L == 0 || (is_pinned(twice_h1) && is_pinned(twice_h2) && is_pinned(valid_mask));
    RunParams rp{minlen, support, unphased, twice_h1, twice_h2, valid_mask, ctx->opt_timing};
    if (!direct_out) {
        const size_t need = (size_t)L * 17 + 64;
        if (need > ctx->h_stage_bytes) {
            if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
            ctx->h_stage = nullptr;
            ctx->h_stage_bytes = 0;
            CU_TRY(ctx, cudaMallocHost(&ctx->h_stage, need));
            ctx->h_stage_bytes = need;
        }
        rp.o1 = static_cast<int64_t *>(ctx->h_stage);
        rp.o2 = rp.o1 + L;
        rp.ov = reinterpret_cast<uint8_t *>(rp.o2 + L);
    }

    if (L) {
        void *a = nullptr, *b = nullptr, *c = nullptr;
        if (cudaHostGetDevicePointer(&a, rp.o1, 0) == cudaSuccess && cudaHostGetDevicePointer(&b, rp.o2, 0) == cudaSuccess &&
            cudaHostGetDevicePointer(&c, rp.ov, 0) == cudaSuccess) {
            rp.d1 = static_cast<int64_t *>(a);
            rp.d2 = static_cast<int64_t *>(b);
            rp.dv = static_cast<uint8_t *>(c);
        } else {
            cudaGetLastError();                               // pinned but not mapped: the copy engines take it
        }
    }

    // the call buffer holds one slot per candidate; on the first call of a context its size is read back from a
    // join-only pre-pass, afterwards it is sized from the previous run and checked after the pass
    if (work && ctx->vals.cap == 0) {
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_ctr, 0, sizeof(DevCounters), s));
        CU_TRY(ctx, cudaMemsetAsync(ctx->delta.p, 0, ((uint64_t)L + 2) * sizeof(uint32_t), s));
        CU_TRY(ctx, cudaMemsetAsync(ctx->desc_scan.p, 0, 2 * ((uint64_t)loc_scan_tiles(L) + 1) * sizeof(uint64_t), s));
        TRY(launch_join(ctx, unphased, s));
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_total, ctx->seg_off.p + L, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU_TRY(ctx, cudaStreamSynchronize(s));
        TRY(ensure_vals(ctx, (uint64_t)*ctx->h_total + 1));
    }

    uint32_t launches = 0, passes = 0;
    bool used_graph = false, done = false;
    for (int attempt = 0; attempt < 4 && !done; ++attempt) {
        const GraphKey key{ctx->data_gen, ctx->buf_gen, minlen, support, unphased, rp.timing, rp.o1, rp.o2, rp.ov, wide_keys(ctx)};
        ++passes;
        used_graph = false;
        if (ctx->graph && !(ctx->graph_key == key)) drop_graph(ctx);
        if (ctx->opt_graph && !ctx->graph && ctx->have_last_key && ctx->last_key == key) {
            // second call with the same shape: capture the DAG once, replay it from now on
            cudaGraph_t g = nullptr;
            CU_TRY(ctx, cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
            const int rc = enqueue_pass(ctx, rp, true, &ctx->graph_launches);
            cudaError_t e = cudaStreamEndCapture(s, &g);
            if (rc != INQ_OK) { if (g) cudaGraphDestroy(g); return rc; }
            if (e != cudaSuccess) return fail(ctx, INQ_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
            // the nodes keep the priorities of the streams they were captured from (without the flag, every node runs at
            // the priority of S0, which the graph is launched into)
            e = cudaGraphInstantiateWithFlags(&ctx->graph, g, cudaGraphInstantiateFlagUseNodePriority);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) { ctx->graph = nullptr; return fail(ctx, INQ_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
            ctx->graph_key = key;
        }
        if (rp.timing >= 1) CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_START], s));
        if (ctx->graph) {
            CU_TRY(ctx, cudaGraphLaunch(ctx->graph, s));
            launches = ctx->graph_launches;
            used_graph = true;
        } else {
            TRY(enqueue_pass(ctx, rp, false, &launches));
        }
        if (rp.timing >= 1) CU_TRY(ctx, cudaEventRecord(ctx->ev[EV_END], s));
        ctx->last_key = key;
        ctx->have_last_key = true;
        {
            // a blocking synchronize wakes the host tens of microseconds late; a pass takes 0.1 - 3 ms, so poll first
            cudaError_t q = cudaErrorNotReady;
            for (int spin = 0; spin < 200000 && (q = cudaStreamQuery(s)) == cudaErrorNotReady; ++spin) {}
            if (q != cudaSuccess && q != cudaErrorNotReady) CU_TRY(ctx, q);
            CU_TRY(ctx, cudaStreamSynchronize(s));
        }

        const unsigned f = ctx->h_ctr->flags;
        bool retry = false;
        if (f & kFlagEventOverflow) {
            // the event buffers were sized speculatively; the scan still counted every event and slot
            const uint64_t need_raw = ctx->h_ctr->ev_alloc + raw_slack;
            release(ctx->evraw);
            TRY(ensure(ctx, ctx->evraw, need_raw));
            retry = true;
        }
        if (f & kFlagWideCall) {
            // a call outside 30 bits: the medians of this pass are incomplete; these reads take 64-bit keys from now on
            ctx->wide_gen = ctx->data_gen;
            retry = true;
        }
        if (work && (uint64_t)*ctx->h_total + 1 > vals_keys(ctx)) {
            release(ctx->vals);
            TRY(ensure_vals(ctx, (uint64_t)*ctx->h_total + 1));
            retry = true;
        }
        if (retry) { ctx->have_last_key = false; continue; }       // buffers moved: the next attempt launches directly
        if (ctx->plan.big_known) {
            // a chunk whose CTA-path kernel was left out turned out to have deep loci (other parameters than the pass the
            // guess came from): run again with it
            bool again = false;
            for (int c = 0; c < ctx->plan.n_chunks; ++c)
                if (ctx->h_ctr->big_count[c] && !ctx->plan.need_big[c]) { ctx->plan.need_big[c] = true; again = true; }
            if (again) { drop_graph(ctx); ctx->have_last_key = false; continue; }
        }
        if (f & kFlagCountOverflow) return fail(ctx, INQ_ERR_TOO_LARGE, "pair or event count exceeds 2^32");
        if (f & kFlagValsOverflow) return fail(ctx, INQ_ERR_STATE, "internal: call buffer overflow");
        if (f & kFlagBadSa)
            return fail(ctx, INQ_ERR_BAD_SA, "read %llu passes the filter and has a soft clip, but its SA tag is not a string or cannot be split/parsed "
                        "(the reference panics in is_accidental_2d, call.rs:431,439-450)", (unsigned long long)ctx->h_ctr->bad_sa_read);
        if (f & kFlagBadHp)
            return fail(ctx, INQ_ERR_BAD_HP, "read %llu passes the phased filter but carries HP %u, outside {0,1,2} (the reference panics, call.rs:358)",
                        (unsigned long long)ctx->h_ctr->bad_hp_read, ctx->h_ctr->bad_hp_value);
        if (f & kFlagMedianEmpty)
            return fail(ctx, INQ_ERR_MEDIAN_EMPTY, "support == 0 with a bucket without usable calls (the reference panics, call.rs:516)");
        if (!ctx->plan.big_known) {
            for (int c = 0; c < ctx->plan.n_chunks; ++c) ctx->plan.need_big[c] = ctx->h_ctr->big_count[c] != 0;
            ctx->plan.big_known = true;
        }
        done = true;
    }
    if (!done) return fail(ctx, INQ_ERR_STATE, "internal: speculative buffers still too small after 4 attempts");
    ctx->last_n_events = (ntiles && L) ? ctx->h_total[3] : 0;      // .y of wt[n_wt]
    if (!direct_out && L) {
        memcpy(twice_h1, rp.o1, (size_t)L * sizeof(int64_t));
        memcpy(twice_h2, rp.o2, (size_t)L * sizeof(int64_t));
        memcpy(valid_mask, rp.ov, (size_t)L);
    }

    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->n_loci = (uint64_t)L;
        stats->n_reads = R;
        stats->n_cigar_words = C;
        auto total = [&](int k) { uint64_t t = 0; for (int i = 0; i < kStatSlots; ++i) t += ctx->h_ctr->stat[i][k]; return t; };
        stats->n_cigar_words_joined = total(ST_WORDS_JOINED);
        stats->n_reads_joined = total(ST_READS_JOINED);
        stats->n_pairs = total(ST_PAIRS);
        stats->n_candidates = total(ST_CANDIDATES);
        stats->n_events = ctx->last_n_events;
        stats->op_visits = total(ST_OP_VISITS);
        stats->n_kernel_launches = launches;
        stats->n_tiles = ntiles;
        stats->n_ranges = 1;
        stats->used_graph = used_graph ? 1u : 0u;
        stats->reads_sorted = ctx->plan.reads_sorted ? 1u : 0u;
        stats->n_median_chunks = (uint32_t)ctx->plan.n_chunks;
        stats->n_passes = passes;
        stats->key_bytes = wide_keys(ctx) ? 8u : 4u;
        if (rp.timing) {
            auto el = [&](int a, int b) { float ms = 0.f; if (cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]) != cudaSuccess) { cudaGetLastError(); ms = 0.f; } return ms; };
            stats->ms_total = el(EV_START, EV_END);
            if (rp.timing >= 2) {
                stats->ms_join = el(EV_START, EV_JOIN);          // memsets + join + segment offsets, under the CIGAR scan
                stats->ms_index = el(EV_START, EV_INDEX);        // ... of which the zeroing kernel
                stats->ms_cigar = el(EV_SCAN0, EV_SCAN1);
                stats->ms_pairs = el(EV_PAIR0, EV_PAIR1);
                // prefix scan over the warp-tile totals (incl. waiting for the join stream)
                stats->ms_fixup = el(EV_SCAN1, EV_PAIR0);
                stats->ms_median = el(EV_MED0, EV_MED1);
                stats->ms_d2h = el(EV_MED1, EV_D2H);
            } else {
                // S0 runs the scan right after the pass starts: start of the pass -> end of the scan
                // (a few us of fork on top of the kernel: the conservative side for a bandwidth figure)
                stats->ms_cigar = el(EV_START, EV_SCAN1);
            }
            stats->ms_scan = el(EV_SCAN1, EV_END);           // what is left exposed after the CIGAR stream is scanned
        }
        stats->ms_h2d = ctx->ms_h2d;
    }
    return INQ_OK;
}

int inq_debug_events(inq_ctx *ctx, uint64_t *n_events, uint32_t *event_pos, int32_t *event_val, uint64_t cap,
                     uint32_t *read_event_off)
{
    if (!ctx) return INQ_ERR_ARG;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t E = ctx->last_n_events, R = ctx->R;
    if (n_events) *n_events = E;
    // the genotyping pass reads events straight from the scan kernel's warp-tile storage; the per-read
    // lists in CIGAR order with absolute anchors are only materialised here
    TRY(ensure(ctx, ctx->ev_off, R + 1));
    if (ctx->events.cap < E + 1) { release(ctx->events); TRY(ensure(ctx, ctx->events, E + 1)); }
    if (E) {
        const uint64_t fix_warps = (R + 1 + 30) / 31;
        k_read_fixup<<<(unsigned)((fix_warps * 32 + 255) / 256), 256, 0, ctx->stream>>>(ctx->unit_off.p, ctx->rs.p, R, ctx->wt.p, ctx->rd_pre.p,
                                                                                       ctx->wt_sbase.p, ctx->evraw.p, ctx->evraw.cap,
                                                                                       ctx->events.p, ctx->events.cap, ctx->ev_off.p, ctx->d_ctr);
        CU_TRY(ctx, cudaGetLastError());
    } else {
        CU_TRY(ctx, cudaMemsetAsync(ctx->ev_off.p, 0, (R + 1) * sizeof(uint32_t), ctx->stream));
    }
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (read_event_off)
        CU_TRY(ctx, cudaMemcpy(read_event_off, ctx->ev_off.p, (R + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    const uint64_t n = std::min(E, cap);
    if (n && (event_pos || event_val)) {
        uint2 *tmp = (uint2 *)malloc(n * sizeof(uint2));
        if (!tmp) return fail(ctx, INQ_ERR_NOMEM, "host allocation failed");
        cudaError_t e = cudaMemcpy(tmp, ctx->events.p, n * sizeof(uint2), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { free(tmp); return fail(ctx, INQ_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e)); }
        for (uint64_t i = 0; i < n; ++i) {
            if (event_pos) event_pos[i] = tmp[i].x;
            if (event_val) event_val[i] = (int32_t)tmp[i].y;
        }
        free(tmp);
    }
    return INQ_OK;
}

}  // extern "C"
