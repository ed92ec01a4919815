// inq_cohort_capi.cu -- extern "C" entry points of include/inqcohort.h (part of libinqcall.so)
#include "../../include/inqcall.h"
#include "../../include/inqcohort.h"
#include "inq_assoc.cuh"
#include "inq_cohort.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

namespace {

thread_local std::string g_cohort_error;

int cfail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_cohort_error = buf;
    return code;
}

struct Guard {                         // frees everything on every exit path
    std::vector<void *> mem;
    cudaStream_t s = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaError_t alloc(void **q, size_t bytes)
    {
        const cudaError_t e = cudaMalloc(q, bytes);
        if (e == cudaSuccess) mem.push_back(*q);
        return e;
    }
    ~Guard()
    {
        for (void *q : mem) cudaFree(q);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (s) cudaStreamDestroy(s);
    }
};

// Calls launch(std::integral_constant<int, P>()) for the padded design width P of inq_assoc's kernels: 4, 8, 16 or 32.
template <class Launch>
void with_width(int P, Launch launch)
{
    switch (P) {
    case 4: launch(std::integral_constant<int, 4>()); break;
    case 8: launch(std::integral_constant<int, 8>()); break;
    case 16: launch(std::integral_constant<int, 16>()); break;
    default: launch(std::integral_constant<int, 32>()); break;
    }
}

#define CC_TRY(call)                                                                            \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) return cfail(INQ_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

}  // namespace

extern "C" {

const char *inq_cohort_last_error(void) { return g_cohort_error.c_str(); }

int inq_outlier(int device, int method, uint64_t n_rows, uint32_t n_cols, const float *values, uint32_t minsize,
                float zscore_cutoff, uint8_t *row_kept, uint64_t *n_hits, uint64_t *hits, uint64_t cap, float *ms_kernel)
{
    using namespace inqc;
    if (n_hits) *n_hits = 0;
    if (ms_kernel) *ms_kernel = 0.f;
    if (method != INQ_OUTLIER_ZSCORE && method != INQ_OUTLIER_DBSCAN) return cfail(INQ_ERR_ARG, "inq_outlier: unknown method %d", method);
    if (n_rows == 0) return INQ_OK;
    if (n_cols == 0) return cfail(INQ_ERR_ARG, "inq_outlier: a row without value columns (the reference panics, outlier.rs:87-91)");
    if (!values || !n_hits || (cap && !hits)) return cfail(INQ_ERR_ARG, "inq_outlier: NULL array");
    if (n_rows > 0xFFFFFFFFull) return cfail(INQ_ERR_TOO_LARGE, "inq_outlier: more than 2^32-1 rows");
    if (method == INQ_OUTLIER_DBSCAN && n_cols > 4096) return cfail(INQ_ERR_TOO_LARGE, "inq_outlier: dbscan supports at most 4096 columns");
    CC_TRY(cudaSetDevice(device));
    Guard g;
    CC_TRY(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking));
    CC_TRY(cudaEventCreate(&g.e0));
    CC_TRY(cudaEventCreate(&g.e1));
    const size_t bytes = (size_t)n_rows * n_cols * sizeof(float);
    void *d_m, *d_kept, *d_hits, *d_ctr;
    CC_TRY(g.alloc(&d_m, bytes));
    CC_TRY(g.alloc(&d_kept, n_rows));
    CC_TRY(g.alloc(&d_hits, std::max<uint64_t>(cap, 1) * sizeof(unsigned long long)));
    CC_TRY(g.alloc(&d_ctr, sizeof(CohortCounters)));
    CC_TRY(cudaMemcpyAsync(d_m, values, bytes, cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(CohortCounters), g.s));
    CC_TRY(cudaEventRecord(g.e0, g.s));
    if (method == INQ_OUTLIER_ZSCORE) {
        const uint32_t stride = n_cols | 1u;
        const size_t res_smem = (size_t)kZResRows * stride * sizeof(float);
        int sms = 0, smem_max = 0;
        CC_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        CC_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
        const size_t per_warp = zw_warp_bytes(n_cols);
        const int zw_warps = (int)std::min<size_t>(kZwMaxWarps, ((size_t)smem_max - 256) / per_warp);
        if (n_cols % 4 == 0 && n_cols <= 32u * kZwMaskWords && zw_warps >= 2) {
            // every warp its own pipeline over groups of 32 rows (bulk async copies, one lane per row)
            const size_t smem = (size_t)zw_warps * per_warp + (size_t)zw_warps * 12 + 128;
            CC_TRY(cudaFuncSetAttribute(k_outlier_zscore_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const uint64_t groups = (n_rows + 31) / 32;
            const unsigned grid = (unsigned)std::min<uint64_t>((groups + zw_warps - 1) / zw_warps, (uint64_t)sms);
            k_outlier_zscore_warp<<<grid, zw_warps * 32, smem, g.s>>>((const float *)d_m, n_rows, n_cols, (float)minsize, zscore_cutoff,
                                                                     (uint8_t *)d_kept, (unsigned long long *)d_hits, cap, (CohortCounters *)d_ctr);
        } else if (res_smem <= 200u * 1024u) {
            // 32 rows fit in shared memory: the matrix is read once
            CC_TRY(cudaFuncSetAttribute(k_outlier_zscore_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)res_smem));
            const unsigned grid = (unsigned)((n_rows + kZResRows - 1) / kZResRows);
            k_outlier_zscore_rows<<<grid, kZResThreads, res_smem, g.s>>>((const float *)d_m, n_rows, n_cols, stride, (float)minsize, zscore_cutoff,
                                                                        (uint8_t *)d_kept, (unsigned long long *)d_hits, cap, (CohortCounters *)d_ctr);
        } else {
        const unsigned grid = (unsigned)((n_rows + kZRows - 1) / kZRows);
        k_outlier_zscore<<<grid, kZRows, 0, g.s>>>((const float *)d_m, n_rows, n_cols, (float)minsize, zscore_cutoff,
                                                   (uint8_t *)d_kept, (unsigned long long *)d_hits, cap, (CohortCounters *)d_ctr);
        }
    } else {
        uint32_t n2 = 32;
        while (n2 < n_cols) n2 <<= 1;
        uint32_t min_points = 0;                              // samples.len().ilog2(), outlier.rs:39
        while ((2ull << min_points) <= n_cols) ++min_points;
        int sms = 0;
        CC_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        // 64..1024 padded columns: one warp per row, sorted in registers (n2 / 32 keys per lane). Otherwise the
        // shared-memory network: one warp for tiny rows, the 128-thread CTA for rows wider than 1024 columns.
        const int ch = (n2 >= 64 && n2 <= 1024) ? (int)(n2 / 32) : 0;
        const size_t nk = ch ? (size_t)n_cols + (n_cols >> 5) + 1 : n_cols;
        const size_t smem = ((size_t)n_cols * 2 + 1 + nk) * sizeof(uint32_t) + 16;   // rng[n], pc[n + 1], key[nk]
        const unsigned threads = n_cols <= 1024 ? 32u : (unsigned)kDbThreads;
        auto launch = [&](auto kernel) -> int {
            int per_sm = 8;
            CC_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CC_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, (int)threads, smem));
            const unsigned grid = (unsigned)std::min<uint64_t>(n_rows, (uint64_t)sms * std::max(per_sm, 1));
            kernel<<<grid, threads, smem, g.s>>>((const float *)d_m, n_rows, n_cols, n2, (float)minsize, min_points,
                                                 (uint8_t *)d_kept, (unsigned long long *)d_hits, cap, (CohortCounters *)d_ctr);
            return INQ_OK;
        };
        int lrc;
        switch (ch) {
        case 2: lrc = launch(k_outlier_dbscan<2>); break;
        case 4: lrc = launch(k_outlier_dbscan<4>); break;
        case 8: lrc = launch(k_outlier_dbscan<8>); break;
        case 16: lrc = launch(k_outlier_dbscan<16>); break;
        case 32: lrc = launch(k_outlier_dbscan<32>); break;
        default: lrc = launch(k_outlier_dbscan<0>); break;
        }
        if (lrc != INQ_OK) return lrc;
    }
    CC_TRY(cudaGetLastError());
    CC_TRY(cudaEventRecord(g.e1, g.s));
    CohortCounters h;
    CC_TRY(cudaMemcpyAsync(&h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost, g.s));
    if (row_kept) CC_TRY(cudaMemcpyAsync(row_kept, d_kept, n_rows, cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaStreamSynchronize(g.s));
    if (ms_kernel) cudaEventElapsedTime(ms_kernel, g.e0, g.e1);
    if (h.no_mode)
        return cfail(INQ_ERR_NO_MODE, "row %llu passes the minsize test but has no positive value: no mode (the reference panics, outlier.rs:144)",
                     ((unsigned long long)h.no_mode_row_hi << 32) | h.no_mode_row_lo);
    *n_hits = h.n_hits;
    const uint64_t n = std::min<uint64_t>(h.n_hits, cap);
    if (n) {
        CC_TRY(cudaMemcpy(hits, d_hits, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
        std::sort(hits, hits + n);                            // (row, column) = the reference's print order
    }
    if (h.n_hits > cap) return cfail(INQ_ERR_HITS_CAP, "inq_outlier: %llu outliers, capacity %llu", (unsigned long long)h.n_hits, (unsigned long long)cap);
    return INQ_OK;
}

int inq_assoc(int device, int model, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
              const double *y, uint32_t n_cov, const double *cov, double *beta, double *se, double *stat, double *p,
              uint32_t *n_used, uint8_t *status, uint8_t *n_iter, float *ms_kernel)
{
    using namespace inqa;
    if (ms_kernel) *ms_kernel = 0.f;
    if (model != INQ_ASSOC_LINEAR && model != INQ_ASSOC_LOGISTIC && model != INQ_ASSOC_FIRTH) return cfail(INQ_ERR_ARG, "inq_assoc: unknown model %d", model);
    if (predictor != INQ_ASSOC_SUM && predictor != INQ_ASSOC_MAX) return cfail(INQ_ERR_ARG, "inq_assoc: unknown predictor %d", predictor);
    if (n_cov > INQ_ASSOC_MAX_COV) return cfail(INQ_ERR_ARG, "inq_assoc: %u covariates (at most %d)", n_cov, INQ_ASSOC_MAX_COV);
    if (n_rows == 0) return INQ_OK;
    if (n_samples == 0) return cfail(INQ_ERR_ARG, "inq_assoc: no samples");
    if (!haps || !y || (n_cov && !cov) || !beta || !se || !stat || !p || !n_used || !status) return cfail(INQ_ERR_ARG, "inq_assoc: NULL array");
    if ((n_rows + kAWarps - 1) / kAWarps > 0x7FFFFFFFull) return cfail(INQ_ERR_TOO_LARGE, "inq_assoc: too many rows");
    for (uint32_t s = 0; s < n_samples; ++s) {
        if (!std::isfinite(y[s])) return cfail(INQ_ERR_ARG, "inq_assoc: trait of sample %u is not a finite number", s);
        if (model != INQ_ASSOC_LINEAR && y[s] != 0.0 && y[s] != 1.0) return cfail(INQ_ERR_ARG, "inq_assoc: logistic trait of sample %u is not 0 or 1", s);
        for (uint32_t c = 0; c < n_cov; ++c)
            if (!std::isfinite(cov[(size_t)s * n_cov + c])) return cfail(INQ_ERR_ARG, "inq_assoc: covariate %u of sample %u is not a finite number", c, s);
    }
    const uint32_t pdim = n_cov + 2;
    const int P = pdim <= 4 ? 4 : pdim <= 8 ? 8 : pdim <= 16 ? 16 : 32;
    // shared design rows [1, covariates centred by their mean, 0 (x), 0 ...]; the linear trait centred by its mean
    std::vector<double> design((size_t)n_samples * P, 0.0), shift(P, 0.0), yc(y, y + n_samples);
    for (uint32_t c = 0; c < n_cov; ++c) {
        double m = 0.0;
        for (uint32_t s = 0; s < n_samples; ++s) m += cov[(size_t)s * n_cov + c];
        shift[1 + c] = m / n_samples;
    }
    for (uint32_t s = 0; s < n_samples; ++s) {
        design[(size_t)s * P] = 1.0;
        for (uint32_t c = 0; c < n_cov; ++c) design[(size_t)s * P + 1 + c] = cov[(size_t)s * n_cov + c] - shift[1 + c];
    }
    if (model == INQ_ASSOC_LINEAR) {
        double m = 0.0;
        for (uint32_t s = 0; s < n_samples; ++s) m += y[s];
        m /= n_samples;
        for (double &v : yc) v -= m;
    }

    CC_TRY(cudaSetDevice(device));
    Guard g;
    CC_TRY(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking));
    CC_TRY(cudaEventCreate(&g.e0));
    CC_TRY(cudaEventCreate(&g.e1));
    const size_t hap_bytes = (size_t)n_rows * 2 * n_samples * sizeof(double);
    void *d_haps, *d_des, *d_shift, *d_y, *d_res, *d_n, *d_st, *d_it;
    CC_TRY(g.alloc(&d_haps, hap_bytes));
    CC_TRY(g.alloc(&d_des, design.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_shift, shift.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_y, n_samples * sizeof(double)));
    CC_TRY(g.alloc(&d_res, (size_t)n_rows * 4 * sizeof(double)));
    CC_TRY(g.alloc(&d_n, (size_t)n_rows * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_st, (size_t)n_rows));
    CC_TRY(g.alloc(&d_it, (size_t)n_rows));
    CC_TRY(cudaMemcpyAsync(d_haps, haps, hap_bytes, cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_des, design.data(), design.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_shift, shift.data(), shift.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_y, yc.data(), n_samples * sizeof(double), cudaMemcpyHostToDevice, g.s));
    double *r = (double *)d_res;
    const AssocOut out{r, r + n_rows, r + 2 * n_rows, r + 3 * n_rows, (uint32_t *)d_n, (uint8_t *)d_st, (uint8_t *)d_it};
    const unsigned grid = (unsigned)((n_rows + kAWarps - 1) / kAWarps);
    const int lg = model == INQ_ASSOC_LOGISTIC, mx = predictor == INQ_ASSOC_MAX;
    const double *dh = (const double *)d_haps, *dd = (const double *)d_des, *ds = (const double *)d_shift, *dy = (const double *)d_y;
    CC_TRY(cudaEventRecord(g.e0, g.s));
    with_width(P, [&](auto width) {
        constexpr int W = decltype(width)::value;
        if (model == INQ_ASSOC_FIRTH) k_assoc_firth<W><<<grid, kAWarps * 32, 0, g.s>>>(dh, n_rows, n_samples, pdim, mx, dd, ds, dy, out);
        else k_assoc<W><<<grid, kAWarps * 32, 0, g.s>>>(dh, n_rows, n_samples, pdim, lg, mx, dd, ds, dy, out);
    });
    CC_TRY(cudaGetLastError());
    CC_TRY(cudaEventRecord(g.e1, g.s));
    CC_TRY(cudaMemcpyAsync(beta, r, n_rows * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(se, r + n_rows, n_rows * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(stat, r + 2 * n_rows, n_rows * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(p, r + 3 * n_rows, n_rows * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(n_used, d_n, n_rows * sizeof(uint32_t), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(status, d_st, n_rows, cudaMemcpyDeviceToHost, g.s));
    if (n_iter) CC_TRY(cudaMemcpyAsync(n_iter, d_it, n_rows, cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaStreamSynchronize(g.s));
    if (ms_kernel) cudaEventElapsedTime(ms_kernel, g.e0, g.e1);
    return INQ_OK;
}

}  // extern "C"
