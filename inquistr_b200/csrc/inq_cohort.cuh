// inq_cohort.cuh -- sm_100a kernels of the cohort `outlier` rows (reference: src/outlier.rs, v0.13.0).
//
// z-score: the reference sums a row's f32 values left to right (outlier.rs:19,22-28), so bit-exact
// parity needs the same order: one thread owns one row and adds sequentially with __fadd_rn / __fmul_rn
// (never contracted to FMA); the CTA stages 32-column tiles through shared memory so that global loads
// stay coalesced although consecutive threads own consecutive rows.
// dbscan: one CTA per row; sort, then the order-independent form of dbscan 0.3.1 in one dimension:
// core(i) = #{j : |x_i - x_j| < eps} >= min_points, noise(i) = !core(i) && no core point within eps.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace inqc {

struct CohortCounters {
    unsigned long long n_hits;
    unsigned int no_mode;              // a kept row had no positive value (dbscan)
    unsigned int no_mode_row_lo, no_mode_row_hi;
};

constexpr int kZRows = 128;            // rows (= threads) per CTA
constexpr int kZTile = 32;             // columns per shared-memory tile
constexpr int kZHitBuf = 1024;         // outliers buffered per CTA before they are written out

__device__ __forceinline__ float clean(float v) { return (v != v) ? 0.0f : v; }   // outlier.rs:81-84

// Fallback for rows too wide for the resident kernel below: a CTA walks its 128 rows in tiles of 32 columns,
// three passes over global memory / L2. A warp fetches 32 row segments of 128 bytes (coalesced) into
// registers, all loads issued back to back, before the first store to shared memory.
constexpr uint32_t kZWarps = kZRows / 32, kZPerWarp = kZRows / kZWarps;

struct TileRegs { float v[kZPerWarp]; };

__device__ __forceinline__ void fetch_tile(const float *__restrict__ m, uint64_t n_rows, uint32_t n_cols, uint64_t row0,
                                           uint32_t c0, TileRegs &t)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t c = c0 + lane;
#pragma unroll
    for (uint32_t k = 0; k < kZPerWarp; ++k) {
        const uint64_t row = row0 + warp * kZPerWarp + k;
        t.v[k] = (row < n_rows && c < n_cols) ? __ldg(m + row * n_cols + c) : 0.0f;
    }
}
__device__ __forceinline__ void store_tile(const TileRegs &t, float (*tile)[kZTile + 1])
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (uint32_t k = 0; k < kZPerWarp; ++k) tile[warp * kZPerWarp + k][lane] = clean(t.v[k]);   // NaN -> 0 (outlier.rs:81-84)
}

__global__ void __launch_bounds__(kZRows)
k_outlier_zscore(const float *__restrict__ m, uint64_t n_rows, uint32_t n_cols, float minsize, float cutoff,
                 uint8_t *__restrict__ row_kept, unsigned long long *__restrict__ hits, uint64_t cap,
                 CohortCounters *__restrict__ ctr)
{
    __shared__ float tile[kZRows][kZTile + 1];
    __shared__ float s_mean[kZRows], s_sd[kZRows];
    __shared__ uint8_t s_kept[kZRows];
    // outliers of the CTA's rows are collected here and leave with ONE global atomic; overflow falls back
    // to one atomic per outlier
    __shared__ unsigned long long s_hits[kZHitBuf];
    __shared__ unsigned int s_nhits;
    __shared__ unsigned long long s_base;
    if (threadIdx.x == 0) s_nhits = 0;
    const uint64_t row0 = (uint64_t)blockIdx.x * kZRows, row = row0 + threadIdx.x;
    TileRegs regs;
    // pass 1: sequential f32 sum and the maximum (outlier.rs:19, 87-90)
    float sum = 0.0f, mx = 0.0f;
    for (uint32_t c0 = 0; c0 < n_cols; c0 += kZTile) {
        fetch_tile(m, n_rows, n_cols, row0, c0, regs);
        __syncthreads();
        store_tile(regs, tile);
        __syncthreads();
        const uint32_t n = min((uint32_t)kZTile, n_cols - c0);
        for (uint32_t c = 0; c < n; ++c) {
            const float v = tile[threadIdx.x][c];
            sum = __fadd_rn(sum, v);
            mx = (c0 + c == 0 || !(v < mx)) ? v : mx;
        }
    }
    const float count = (float)n_cols;
    const float mean = __fdiv_rn(sum, count);
    const bool kept = row < n_rows && !(mx < minsize);
    // pass 2: population variance around the f32 mean (outlier.rs:22-29)
    float var = 0.0f;
    for (uint32_t c0 = 0; c0 < n_cols; c0 += kZTile) {
        fetch_tile(m, n_rows, n_cols, row0, c0, regs);
        __syncthreads();
        store_tile(regs, tile);
        __syncthreads();
        const uint32_t n = min((uint32_t)kZTile, n_cols - c0);
        for (uint32_t c = 0; c < n; ++c) {
            const float diff = __fsub_rn(mean, tile[threadIdx.x][c]);
            var = __fadd_rn(var, __fmul_rn(diff, diff));
        }
    }
    const float sd = __fsqrt_rn(__fdiv_rn(var, count));
    s_mean[threadIdx.x] = mean;
    s_sd[threadIdx.x] = sd;
    s_kept[threadIdx.x] = kept ? 1 : 0;
    if (row < n_rows && row_kept) row_kept[row] = kept ? 1 : 0;
    __syncthreads();
    // pass 3: flags, element-parallel straight from the registers (no order dependence):
    // (v - mean) / sd >= cutoff (outlier.rs:109)
    {
        const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (uint32_t c0 = 0; c0 < n_cols; c0 += kZTile) {
            fetch_tile(m, n_rows, n_cols, row0, c0, regs);
            const uint32_t c = c0 + lane;
#pragma unroll
            for (uint32_t k = 0; k < kZPerWarp; ++k) {
                const uint32_t r = warp * kZPerWarp + k;
                if (!s_kept[r] || c >= n_cols) continue;
                const float z = __fdiv_rn(__fsub_rn(clean(regs.v[k]), s_mean[r]), s_sd[r]);
                if (z >= cutoff) {
                    const unsigned long long h = ((row0 + r) << 32) | c;
                    const unsigned int slot_l = atomicAdd(&s_nhits, 1u);
                    if (slot_l < (unsigned int)kZHitBuf) s_hits[slot_l] = h;
                    else {
                        const unsigned long long slot = atomicAdd(&ctr->n_hits, 1ull);
                        if (slot < cap) hits[slot] = h;
                    }
                }
            }
        }
    }
    __syncthreads();
    const unsigned int nh = min(s_nhits, (unsigned int)kZHitBuf);
    if (threadIdx.x == 0 && nh) s_base = atomicAdd(&ctr->n_hits, (unsigned long long)nh);
    __syncthreads();
    for (unsigned int k = threadIdx.x; k < nh; k += blockDim.x)
        if (s_base + k < cap) hits[s_base + k] = s_hits[k];
}

// ---------------------------------------------------------------------------------------------- z-score, resident rows
// When 32 rows fit in shared memory (n_cols <= ~1700) the matrix is read from HBM exactly once: the CTA copies
// its 32 contiguous rows in (coalesced, all 256 threads), one warp then owns one row per lane and does the two
// order-dependent passes out of shared memory (odd row stride: conflict-free), and all threads take the
// element-parallel flag pass. Several CTAs per SM overlap one CTA's copy with another's sums.
constexpr int kZResRows = 32;
constexpr int kZResThreads = 256;
constexpr int kZResHitBuf = 512;

// (v - mean) / sd >= cutoff with the reference's f32 division (outlier.rs:109). The correctly rounded division
// is only evaluated when the reciprocal-multiply estimate is within 1e-5 (relative) of the cutoff or not finite;
// the estimate is off by < 2e-7 relative, so everywhere else it decides identically.
__device__ __forceinline__ bool z_at_least(float d, float sd, float rinv, float cutoff, float margin)
{
    const float zp = d * rinv;
    if (fabsf(zp - cutoff) > margin && fabsf(zp) <= 3.0e38f) return zp > cutoff;
    return __fdiv_rn(d, sd) >= cutoff;
}

__global__ void __launch_bounds__(kZResThreads)
k_outlier_zscore_rows(const float *__restrict__ m, uint64_t n_rows, uint32_t n_cols, uint32_t stride, float minsize,
                      float cutoff, uint8_t *__restrict__ row_kept, unsigned long long *__restrict__ hits, uint64_t cap,
                      CohortCounters *__restrict__ ctr)
{
    extern __shared__ float zr_rows[];                       // [kZResRows][stride], stride odd
    __shared__ float s_mean[kZResRows], s_sd[kZResRows], s_rinv[kZResRows];
    __shared__ uint8_t s_kept[kZResRows];
    __shared__ unsigned long long s_hits[kZResHitBuf];
    __shared__ unsigned int s_nhits;
    __shared__ unsigned long long s_base;
    const uint32_t tid = threadIdx.x;
    if (tid == 0) s_nhits = 0;
    const uint64_t row0 = (uint64_t)blockIdx.x * kZResRows;
    const uint32_t nr = (uint32_t)min((uint64_t)kZResRows, n_rows - row0);
    const float *__restrict__ src = m + row0 * n_cols;
    // ---- copy in (NaN -> 0, outlier.rs:81-84): a warp takes rows w, w + 8, ...; its lanes stride over the row's
    //      columns (coalesced 128-byte requests), up to 16 loads per lane in flight before the first store
    const uint32_t lane = tid & 31, warp = tid >> 5;
    constexpr uint32_t kWarps = kZResThreads / 32;
    for (uint32_t r = warp; r < nr; r += kWarps) {
        const float *__restrict__ g = src + (size_t)r * n_cols;
        float *row = zr_rows + r * stride;
        for (uint32_t c0 = 0; c0 < n_cols; c0 += 32 * 16) {
            float v[16];
#pragma unroll
            for (uint32_t k = 0; k < 16; ++k) {
                const uint32_t c = c0 + k * 32 + lane;
                v[k] = c < n_cols ? __ldg(g + c) : 0.0f;
            }
#pragma unroll
            for (uint32_t k = 0; k < 16; ++k) {
                const uint32_t c = c0 + k * 32 + lane;
                if (c < n_cols) row[c] = clean(v[k]);
            }
        }
    }
    __syncthreads();
    // ---- one lane per row: sequential f32 sum + max, then the population variance (outlier.rs:18-31,87-90)
    if (tid < nr) {
        const float *row = zr_rows + tid * stride;
        float sum = 0.0f, mx = -INFINITY;
#pragma unroll 16
        for (uint32_t c = 0; c < n_cols; ++c) {             // unrolled: the shared-memory loads run ahead of the add chain
            const float v = row[c];
            sum = __fadd_rn(sum, v);
            mx = fmaxf(mx, v);
        }
        const float count = (float)n_cols;
        const float mean = __fdiv_rn(sum, count);
        float var = 0.0f;
#pragma unroll 16
        for (uint32_t c = 0; c < n_cols; ++c) {
            const float diff = __fsub_rn(mean, row[c]);
            var = __fadd_rn(var, __fmul_rn(diff, diff));
        }
        const float sd = __fsqrt_rn(__fdiv_rn(var, count));
        const bool kept = !(mx < minsize);
        s_mean[tid] = mean;
        s_sd[tid] = sd;
        s_rinv[tid] = __frcp_rn(sd);
        s_kept[tid] = kept ? 1 : 0;
        if (row_kept) row_kept[row0 + tid] = kept ? 1 : 0;
    }
    __syncthreads();
    // ---- flags, element-parallel
    {
        const float margin = fabsf(cutoff) * 1e-5f + 1e-30f;
        for (uint32_t r = warp; r < nr; r += kWarps) {
            if (!s_kept[r]) continue;
            const float mean = s_mean[r], sd = s_sd[r], rinv = s_rinv[r];
            const float *row = zr_rows + r * stride;
            for (uint32_t c = lane; c < n_cols; c += 32) {
                if (z_at_least(__fsub_rn(row[c], mean), sd, rinv, cutoff, margin)) {
                    const unsigned long long h = ((row0 + r) << 32) | c;
                    const unsigned int k = atomicAdd(&s_nhits, 1u);
                    if (k < (unsigned int)kZResHitBuf) s_hits[k] = h;
                    else {
                        const unsigned long long slot = atomicAdd(&ctr->n_hits, 1ull);
                        if (slot < cap) hits[slot] = h;
                    }
                }
            }
        }
    }
    __syncthreads();
    const unsigned int nh = min(s_nhits, (unsigned int)kZResHitBuf);
    if (tid == 0 && nh) s_base = atomicAdd(&ctr->n_hits, (unsigned long long)nh);
    __syncthreads();
    for (unsigned int k = tid; k < nh; k += kZResThreads)
        if (s_base + k < cap) hits[s_base + k] = s_hits[k];
}

// ---------------------------------------------------------------------------------------------- z-score, warp-autonomous
// The order-dependent sums are one lane per row, so every lane of every warp has to own a row for the SM to be busy:
// each warp is its own pipeline over groups of 32 consecutive rows. Lane k issues ONE bulk async copy (TMA,
// cp.async.bulk) of row k into the warp's private slab and the warp waits on its own mbarrier -- no registers and
// no issue slots are spent on the copy, and while one warp of the SM waits for its rows the others add. The rows
// sit `stride` words apart with stride = 4 * odd, which makes the per-lane LDS.128 of the two sequential passes
// conflict-free (8 lanes x 16 bytes hit 8 different 4-bank groups). The flag pass is a third lane-per-row pass that
// leaves one bit per column; one global atomic per group reserves the output slots. The matrix is read from HBM exactly once.
// Needs n_cols % 4 == 0 (16-byte aligned rows) -- other shapes take k_outlier_zscore_rows.
constexpr int kZwMaskWords = 33;          // u32 hit-mask words per lane (odd stride): rows of up to 1056 columns take the fast flag pass
constexpr int kZwMaxWarps = 16;

__device__ __forceinline__ uint32_t zw_smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__host__ __device__ inline uint32_t zw_stride(uint32_t n_cols) { return ((n_cols / 4) & 1u) ? n_cols : n_cols + 4; }
__host__ __device__ inline size_t zw_warp_bytes(uint32_t n_cols) { return (size_t)32 * zw_stride(n_cols) * 4 + (size_t)32 * kZwMaskWords * 4; }

__global__ void __launch_bounds__(kZwMaxWarps * 32, 1)
k_outlier_zscore_warp(const float *__restrict__ m, uint64_t n_rows, uint32_t n_cols, float minsize, float cutoff,
                      uint8_t *__restrict__ row_kept, unsigned long long *__restrict__ hits, uint64_t cap,
                      CohortCounters *__restrict__ ctr)
{
    extern __shared__ __align__(128) unsigned char zw_smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const uint32_t stride = zw_stride(n_cols);
    float *rows = reinterpret_cast<float *>(zw_smem + (size_t)warp * zw_warp_bytes(n_cols));
    uint64_t *bar = reinterpret_cast<uint64_t *>(zw_smem + (size_t)nwarps * zw_warp_bytes(n_cols)) + warp;
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(zw_smem_u32(bar)), "r"(1) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const uint64_t n_groups = (n_rows + 31) / 32;
    const uint32_t row_bytes = n_cols * 4u;
    const float count = (float)n_cols;
    const float margin = fabsf(cutoff) * 1e-5f + 1e-30f;
    uint32_t parity = 0;
    for (uint64_t g = (uint64_t)blockIdx.x * nwarps + warp; g < n_groups; g += (uint64_t)gridDim.x * nwarps) {
        const uint64_t row0 = g * 32;
        const uint32_t nr = (uint32_t)min((uint64_t)32, n_rows - row0);
        // ---- rows in: one bulk copy per lane, all on the warp's mbarrier
        if (lane == 0)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(zw_smem_u32(bar)), "r"(nr * row_bytes) : "memory");
        __syncwarp();
        if (lane < nr)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(zw_smem_u32(rows + lane * stride)), "l"(m + (row0 + lane) * n_cols), "r"(row_bytes), "r"(zw_smem_u32(bar))
                         : "memory");
        {
            uint32_t done = 0;
            while (true) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(done) : "r"(zw_smem_u32(bar)), "r"(parity) : "memory");
                if (done) break;
                __nanosleep(64);
            }
            parity ^= 1u;
        }
        // ---- one lane per row: sequential f32 sum + max, then the population variance (outlier.rs:18-31,81-90)
        float mean = 0.0f, sd = 0.0f, rinv = 0.0f;
        bool kept = false;
        if (lane < nr) {
            const float4 *row4 = reinterpret_cast<const float4 *>(rows + lane * stride);
            float sum = 0.0f, mx = -INFINITY;
#pragma unroll 4
            for (uint32_t c = 0; c < n_cols / 4; ++c) {
                const float4 v = row4[c];
                const float a = clean(v.x), b = clean(v.y), d = clean(v.z), e = clean(v.w);     // NaN -> 0
                sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, a), b), d), e);
                mx = fmaxf(fmaxf(mx, fmaxf(a, b)), fmaxf(d, e));
            }
            mean = __fdiv_rn(sum, count);
            float var = 0.0f;
#pragma unroll 4
            for (uint32_t c = 0; c < n_cols / 4; ++c) {
                const float4 v = row4[c];
                const float da = __fsub_rn(mean, clean(v.x)), db = __fsub_rn(mean, clean(v.y));
                const float dc = __fsub_rn(mean, clean(v.z)), dd = __fsub_rn(mean, clean(v.w));
                var = __fadd_rn(var, __fmul_rn(da, da));
                var = __fadd_rn(var, __fmul_rn(db, db));
                var = __fadd_rn(var, __fmul_rn(dc, dc));
                var = __fadd_rn(var, __fmul_rn(dd, dd));
            }
            sd = __fsqrt_rn(__fdiv_rn(var, count));
            rinv = __frcp_rn(sd);
            kept = !(mx < minsize);
            if (row_kept) row_kept[row0 + lane] = kept ? 1 : 0;
        }
        // ---- flags (outlier.rs:99-113): still one lane per row -- a third pass with the same conflict-free LDS.128 that
        //      leaves one bit per column in the lane's mask words. (A row-major, element-parallel pass leaves this single
        //      warp with one dependent load -> test -> vote chain per 32 columns and nothing to hide it behind: measured
        //      0.96 ms of 1.08; a data-dependent branch per load costs the full LDS latency every time: 0.135 ms for the
        //      pass without a single hit. Hence: branch-free mask build, then the set bits are enumerated.)
        uint32_t *bits = reinterpret_cast<uint32_t *>(rows + 32 * stride) + lane * kZwMaskWords;
        const uint32_t n4 = n_cols / 4, nwords = (n4 + 7) / 8;
        uint32_t cnt = 0;
        if (lane < nr && kept) {
            const float4 *row4 = reinterpret_cast<const float4 *>(rows + lane * stride);
            // The reference's test fl(fl(v - mean) / sd) >= cutoff (outlier.rs:109) is a step function of v: both roundings
            // are monotone for sd > 0. Its exact threshold -- the smallest f32 that passes -- is found once per row by
            // walking a few ulps from mean + cutoff * sd with the real predicate; the pass then costs one compare per value
            // instead of a subtract, a divide estimate and three compares. Rows where that does not apply (sd not positive
            // and finite, or the walk does not settle) use the predicate itself.
            bool have_thr = false;
            float thr = 0.0f;
            if (sd > 0.0f && sd <= 3.0e38f && fabsf(mean) <= 3.0e38f && fabsf(cutoff) <= 3.0e38f) {
                auto pred = [&](float v) { return __fdiv_rn(__fsub_rn(v, mean), sd) >= cutoff; };
                auto step = [](float v, bool up) {               // next representable f32 above / below (finite v)
                    uint32_t u = __float_as_uint(v);
                    if ((u << 1) == 0u) return __uint_as_float(up ? 0x00000001u : 0x80000001u);
                    const bool neg = (u >> 31) != 0u;
                    u += (up != neg) ? 1u : 0xFFFFFFFFu;
                    return __uint_as_float(u);
                };
                float t = __fmaf_rn(cutoff, sd, mean);
                if (fabsf(t) <= 3.0e38f) {
                    int guard = 0;
                    if (pred(t)) {
                        for (; guard < 16; ++guard) { const float d = step(t, false); if (!(fabsf(d) <= 3.0e38f) || !pred(d)) break; t = d; }
                    } else {
                        for (; guard < 16; ++guard) { t = step(t, true); if (!(fabsf(t) <= 3.0e38f) || pred(t)) break; }
                    }
                    have_thr = guard < 16 && fabsf(t) <= 3.0e38f && pred(t) && !pred(step(t, false));
                    thr = t;
                }
            }
            if (have_thr) {
                for (uint32_t w = 0; w < nwords; ++w) {
                    uint32_t acc = 0;
#pragma unroll
                    for (uint32_t j = 0; j < 8; ++j) {
                        const uint32_t c = w * 8 + j;
                        float4 v = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
                        if (c < n4) v = row4[c];
                        const uint32_t m = (clean(v.x) >= thr ? 1u : 0u) | (clean(v.y) >= thr ? 2u : 0u) | (clean(v.z) >= thr ? 4u : 0u) |
                                           (clean(v.w) >= thr ? 8u : 0u);
                        acc |= m << (4 * j);
                    }
                    bits[w] = acc;
                    cnt += __popc(acc);
                }
            } else {
                const float *row = rows + lane * stride;
                for (uint32_t w = 0; w < nwords; ++w) {
                    uint32_t acc = 0;
                    for (uint32_t j = 0; j < 32 && 32 * w + j < n_cols; ++j)
                        if (z_at_least(__fsub_rn(clean(row[32 * w + j]), mean), sd, rinv, cutoff, margin)) acc |= 1u << j;
                    bits[w] = acc;
                    cnt += __popc(acc);
                }
            }
        }
        // one global atomic per group reserves the slots; every lane writes its own row's hits (the host sorts them)
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if ((int)lane >= d) incl += o; }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (total) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&ctr->n_hits, (unsigned long long)total);
            unsigned long long slot = __shfl_sync(0xffffffffu, base, 0) + (incl - cnt);
            if (cnt) {
                const unsigned long long rowbits = (row0 + lane) << 32;
                for (uint32_t w = 0; w < nwords; ++w) {
                    uint32_t m = bits[w];
                    while (m) {
                        const uint32_t bpos = (uint32_t)__ffs((int)m) - 1u;
                        m &= m - 1u;
                        if (slot < cap) hits[slot] = rowbits | (32u * w + bpos);
                        ++slot;
                    }
                }
            }
        }
        __syncwarp();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // the slab is refilled by the async proxy next
    }
}

// ---------------------------------------------------------------------------------------------- dbscan
constexpr int kDbThreads = 128;

__device__ __forceinline__ uint32_t block_scan_excl(uint32_t v, uint32_t *s_warp, uint32_t *total)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if ((int)lane >= d) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    uint32_t base = 0, tot = 0;
    for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) {
        if (w < warp) base += s_warp[w];
        tot += s_warp[w];
    }
    __syncthreads();
    *total = tot;
    return base + x - v;
}

// one CTA per row, two sort engines:
//  * CH == 0 (rows wider than 1024 columns, or narrower than 64): 128 threads (one warp for tiny rows), an
//    all-ascending bitonic network in shared memory over the next power of two with VIRTUAL +inf padding: a
//    comparator whose upper end lies at or beyond n is a no-op, so only the ~n/2 real comparators of a stage are
//    enumerated.
//  * CH  > 0 (n2 = 32 * CH <= 1024): one warp, the whole row in registers, lane-major (element e = lane * CH + k):
//    the 40 of 55 stages whose comparators span fewer than CH elements are min/max pairs on a lane's own
//    registers, the rest exchange with `shfl.xor` — no shared memory, no barrier, no index arithmetic.
// Only the VALUES are sorted (order-preserving u32 image of the f32): in one dimension a point's class depends on
// its value alone, so the columns of the few noise values are recovered at the end by scanning the row for them,
// which is far cheaper than dragging a column index through every comparator.
// Shared memory after the sort: key[] f32 sorted values, pc[n + 1] u32 prefix count of core points, rng[n] u32 each
// element's neighbour range (then the list of noise values). In register mode key[] is written lane-major, so it
// carries one pad slot per 32 elements to keep those stores off a single bank.
__device__ __forceinline__ uint32_t f32_orderable(float v)
{
    const uint32_t u = __float_as_uint(v);
    return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float f32_from_orderable(uint32_t o)
{
    return __uint_as_float(o ^ ((o >> 31) ? 0x80000000u : 0xFFFFFFFFu));
}

template <bool PAD> struct SortedKeys {
    const float *key;
    __device__ __forceinline__ float operator[](uint32_t i) const { return key[PAD ? i + (i >> 5) : i]; }
};

// neighbours of sorted element i: the contiguous run [lo, hi) with |key[i] - key[j]| < eps, decided in f64
// like dbscan's euclidean distance (range_query's `distance < eps`). The binary searches run on f32 thresholds
// rounded towards the side that keeps them exact for an exact x -+ eps (key > T <=> key > rd(T); key >= U <=>
// key >= ru(U)); the f64 predicate itself then settles the boundary, so a difference that rounds in f64 still
// lands where the reference's comparison puts it.
template <bool PAD>
__device__ __forceinline__ void eps_range(const SortedKeys<PAD> key, uint32_t n, uint32_t i, double eps, uint32_t *lo, uint32_t *hi)
{
    const double x = (double)key[i];
    const float tg = __double2float_rd(x - eps);
    uint32_t a = 0, b = i;                               // first j <= i with x - key[j] < eps
    while (a < b) { const uint32_t mid = (a + b) >> 1; if (!(key[mid] > tg)) a = mid + 1; else b = mid; }
    while (a > 0 && (x - (double)key[a - 1] < eps)) --a;
    while (a < i && !(x - (double)key[a] < eps)) ++a;
    *lo = a;
    const float uf = __double2float_ru(x + eps);
    a = i; b = n;                                        // first j >= i with key[j] - x >= eps
    while (a < b) { const uint32_t mid = (a + b) >> 1; if (key[mid] < uf) a = mid + 1; else b = mid; }
    while (a > i && !((double)key[a - 1] - x < eps)) --a;
    while (a < n && ((double)key[a] - x < eps)) ++a;
    *hi = a;
}

__device__ __forceinline__ void cmpswap(uint32_t &lo, uint32_t &hi)
{
    const uint32_t a = lo, b = hi;
    lo = min(a, b);
    hi = max(a, b);
}
// this lane keeps the smaller or (upper) the larger of its own and its partner's key: one predicated VIMNMX
__device__ __forceinline__ uint32_t keep_of(uint32_t mine, uint32_t other, bool upper)
{
    return upper ? max(mine, other) : min(mine, other);
}

template <int CH>
__device__ __forceinline__ void warp_sort(uint32_t (&r)[CH], uint32_t lane)
{
#pragma unroll
    for (int blk = 2; blk <= CH * 32; blk <<= 1) {
        // mirror step: element i meets i ^ (blk - 1)
        if (blk <= CH) {
#pragma unroll
            for (int k = 0; k < CH; ++k)
                if ((k ^ (blk - 1)) > k) cmpswap(r[k], r[k ^ (blk - 1)]);
        } else {
            const int lm = blk / CH - 1;                     // partner lane = lane ^ lm, partner slot = CH - 1 - k
            const bool upper = (lane & (uint32_t)(blk / CH / 2)) != 0;
#pragma unroll
            for (int k = 0; k < CH / 2; ++k) {
                const uint32_t pa = __shfl_xor_sync(0xffffffffu, r[CH - 1 - k], lm);
                const uint32_t pb = __shfl_xor_sync(0xffffffffu, r[k], lm);
                r[k] = keep_of(r[k], pa, upper);
                r[CH - 1 - k] = keep_of(r[CH - 1 - k], pb, upper);
            }
        }
        // half-cleaners: element i (bit d clear) meets i + d
#pragma unroll
        for (int d = blk / 4; d >= 1; d >>= 1) {
            if (d >= CH) {
                const bool upper = (lane & (uint32_t)(d / CH)) != 0;
#pragma unroll
                for (int k = 0; k < CH; ++k) r[k] = keep_of(r[k], __shfl_xor_sync(0xffffffffu, r[k], d / CH), upper);
            } else {
#pragma unroll
                for (int k = 0; k < CH; ++k)
                    if ((k & d) == 0) cmpswap(r[k], r[k + d]);
            }
        }
    }
}

template <int CH>
__global__ void __launch_bounds__(CH ? 32 : kDbThreads)
k_outlier_dbscan(const float *__restrict__ m, uint64_t n_rows, uint32_t n_cols, uint32_t n2, float minsize,
                 uint32_t min_points, uint8_t *__restrict__ row_kept, unsigned long long *__restrict__ hits,
                 uint64_t cap, CohortCounters *__restrict__ ctr)
{
    constexpr bool PAD = CH > 0;
    constexpr int CHR = CH ? CH : 1;
    extern __shared__ __align__(8) unsigned char db_smem[];
    const uint32_t n = n_cols;
    const uint32_t nk = PAD ? n + (n >> 5) + 1 : n;        // slots of key[]
    uint32_t *rng = reinterpret_cast<uint32_t *>(db_smem);
    uint32_t *pc = rng + n;
    float *key = reinterpret_cast<float *>(pc + n + 1);
    uint32_t *ukey = reinterpret_cast<uint32_t *>(key);    // CH == 0: the keys are sorted in place as u32 images
    float *noise_val = reinterpret_cast<float *>(rng);     // once the ranges are consumed
    const SortedKeys<PAD> skeys{key};
    __shared__ uint32_t s_warp[kDbThreads / 32];
    __shared__ float s_wmax[kDbThreads / 32];
    __shared__ unsigned long long s_best;
    __shared__ uint32_t s_nnoise;
    const uint32_t tid = threadIdx.x;
    (void)nk;
    for (uint64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const float *mrow = m + row * n_cols;
        __syncthreads();
        if (tid == 0) { s_best = 0ull; s_nnoise = 0u; }
        float mx = -INFINITY;
        uint32_t r[CHR];
        if constexpr (PAD) {
#pragma unroll
            for (int k = 0; k < CHR; ++k) {
                const uint32_t e = tid * CHR + k;
                r[k] = 0xFFFFFFFFu;                          // above every real image (that pattern is a NaN, cleaned to 0)
                if (e < n) {
                    const float v = clean(__ldg(mrow + e));
                    mx = (v > mx) ? v : mx;
                    r[k] = f32_orderable(v);
                }
            }
        } else {
            for (uint32_t i = tid; i < n; i += blockDim.x) {
                const float v = clean(mrow[i]);
                mx = (v > mx) ? v : mx;
                ukey[i] = f32_orderable(v);
            }
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) { const float o = __shfl_xor_sync(0xffffffffu, mx, d); mx = (o > mx) ? o : mx; }
        if ((tid & 31) == 0) s_wmax[tid >> 5] = mx;
        __syncthreads();
        float row_max = s_wmax[0];
        for (uint32_t w = 1; w < (blockDim.x >> 5); ++w) row_max = (s_wmax[w] > row_max) ? s_wmax[w] : row_max;
        const bool kept = !(row_max < minsize);
        if (tid == 0 && row_kept) row_kept[row] = kept ? 1 : 0;
        if (!kept) continue;

        // ---- sort the values
        if constexpr (PAD) {
            warp_sort<CHR>(r, tid);
#pragma unroll
            for (int k = 0; k < CHR; ++k) {
                const uint32_t e = tid * CHR + k;
                if (e < n) key[e + (e >> 5)] = f32_from_orderable(r[k]);
            }
        } else {
            // comparator q of a stage is found with shifts only (blk and d are powers of two)
            for (uint32_t lb = 1; (1u << lb) <= n2; ++lb) {
                const uint32_t blk = 1u << lb;
                // mirror step: comparator q joins i = (q >> (lb-1)) * blk + (q & (h-1)) with j = i ^ (blk - 1), h = blk / 2
                {
                    const uint32_t h = blk >> 1;
                    for (uint32_t q = tid;; q += blockDim.x) {
                        const uint32_t i = ((q >> (lb - 1)) << lb) + (q & (h - 1));
                        if (i >= n) break;
                        const uint32_t j = i ^ (blk - 1);
                        if (j < n) {
                            const uint32_t a = ukey[i], b = ukey[j];
                            if (a > b) { ukey[i] = b; ukey[j] = a; }
                        }
                    }
                    __syncthreads();
                }
                for (int ld = (int)lb - 2; ld >= 0; --ld) {
                    const uint32_t d = 1u << ld;
                    for (uint32_t q = tid;; q += blockDim.x) {
                        const uint32_t i = ((q >> ld) << (ld + 1)) + (q & (d - 1));
                        if (i >= n) break;
                        const uint32_t j = i + d;
                        if (j < n) {
                            const uint32_t a = ukey[i], b = ukey[j];
                            if (a > b) { ukey[i] = b; ukey[j] = a; }
                        }
                    }
                    __syncthreads();
                }
            }
            for (uint32_t i = tid; i < n; i += blockDim.x) key[i] = f32_from_orderable(ukey[i]);
        }
        __syncthreads();

        // ---- mode of `value as usize` over the positive values (outlier.rs:133-145): the sorted order
        //      is also the order of the truncated values, so a run's length is one binary search from its first element.
        //      Ties: the smallest value (the reference's HashMap order is random).
        unsigned long long best = 0ull;                      // (count << 32) | ~rank  -> max = most frequent, then smallest
        for (uint32_t i = tid; i < n_cols; i += blockDim.x) {
            const float v = skeys[i];
            if (!(v > 0.0f)) continue;
            const float t = truncf(v);
            if (i > 0) {                                     // only the first element of a run of equal truncations counts it
                const float p = skeys[i - 1];
                if (p > 0.0f && truncf(p) == t) continue;
            }
            uint32_t lo2 = i + 1, hi2 = n_cols;              // first j whose truncation exceeds t (exact at any magnitude)
            while (lo2 < hi2) { const uint32_t mid = (lo2 + hi2) >> 1; if (truncf(skeys[mid]) <= t) lo2 = mid + 1; else hi2 = mid; }
            const unsigned long long cand = ((unsigned long long)(lo2 - i) << 32) | (0xFFFFFFFFu - i);
            best = cand > best ? cand : best;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, d);
            best = o > best ? o : best;
        }
        if ((tid & 31) == 0 && best) atomicMax(&s_best, best);
        __syncthreads();
        if (s_best == 0ull) {                                // no positive value: the reference panics
            if (tid == 0) {
                atomicExch(&ctr->no_mode, 1u);
                ctr->no_mode_row_lo = (unsigned int)row;
                ctr->no_mode_row_hi = (unsigned int)(row >> 32);
            }
            continue;
        }
        const uint32_t mode_first = 0xFFFFFFFFu - (uint32_t)(s_best & 0xFFFFFFFFull);
        const float mode_f = truncf(skeys[mode_first]);
        // eps = max(2 * mode, 10) as f64 (outlier.rs:118); mode < 2^24 is exact in f32 and doubling is exact in f64
        const double eps = fmax(2.0 * (double)mode_f, 10.0);

        // ---- core points: |x_i - x_j| < eps in f64 (dbscan's euclidean distance), j over the whole row
        for (uint32_t i = tid; i < n; i += blockDim.x) {
            uint32_t lo = 0, hi = 0;
            eps_range(skeys, n_cols, i, eps, &lo, &hi);
            rng[i] = lo | (hi << 16);                        // n_cols <= 4096: both fit 16 bits
            pc[i] = (hi - lo >= min_points) ? 1u : 0u;
        }
        __syncthreads();
        // exclusive prefix count of core points over the sorted order: chunked block scan
        uint32_t carry = 0;
        for (uint32_t base = 0; base < n; base += blockDim.x) {
            const uint32_t i = base + tid;
            const uint32_t v = i < n ? pc[i] : 0u;
            uint32_t tot;
            const uint32_t ex = block_scan_excl(v, s_warp, &tot);
            if (i < n) pc[i] = carry + ex;
            carry += tot;
        }
        if (tid == 0) pc[n] = carry;
        __syncthreads();
        // ---- noise = not core and no core point within eps (Edge otherwise). Equal values share a class, so a
        //      noise VALUE is listed once (by the first element of its run)
        uint32_t mine = 0;                                   // bit q: element tid + q * blockDim.x opens a run of noise values
        for (uint32_t i = tid, q = 0; i < n_cols; i += blockDim.x, ++q) {
            const uint32_t lo = rng[i] & 0xFFFFu, hi = rng[i] >> 16;
            const bool core = hi - lo >= min_points;
            const bool near_core = pc[hi] - pc[lo] > 0u;
            if (!core && !near_core && (i == 0 || !(skeys[i - 1] == skeys[i]))) mine |= 1u << q;
        }
        __syncthreads();                                     // every range is consumed: rng becomes the noise list
        for (uint32_t q = 0; mine; ++q, mine >>= 1)
            if (mine & 1u) noise_val[atomicAdd(&s_nnoise, 1u)] = skeys[tid + q * blockDim.x];
        __syncthreads();
        // ---- the columns holding a noise value are the row's outliers (host sorts the (row, column) list)
        const uint32_t nn = s_nnoise;
        for (uint32_t w = 0; w < nn; ++w) {
            const float v = noise_val[w];
            for (uint32_t c = tid; c < n_cols; c += blockDim.x)
                if (clean(__ldg(mrow + c)) == v) {
                    const unsigned long long slot = atomicAdd(&ctr->n_hits, 1ull);
                    if (slot < cap) hits[slot] = (row << 32) | c;
                }
        }
    }
}

}  // namespace inqc
