// inq_cohort_capi.cu -- extern "C" entry points of include/inqcohort.h (part of libinqcall.so)
#include "../../include/inqcall.h"
#include "../../include/inqcohort.h"
#include "inq_assoc.cuh"
#include "inq_cohort.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstdint>
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

// ---- assoc: the checks and the host preparation shared by inq_assoc and inq_assoc_traits

int assoc_width(uint32_t pdim) { return pdim <= 4 ? 4 : pdim <= 8 ? 8 : pdim <= 16 ? 16 : 32; }

int assoc_check_args(const char *fn, int model, int predictor, uint32_t n_cov)
{
    if (model != INQ_ASSOC_LINEAR && model != INQ_ASSOC_LOGISTIC && model != INQ_ASSOC_FIRTH) return cfail(INQ_ERR_ARG, "%s: unknown model %d", fn, model);
    if (predictor != INQ_ASSOC_SUM && predictor != INQ_ASSOC_MAX) return cfail(INQ_ERR_ARG, "%s: unknown predictor %d", fn, predictor);
    if (n_cov > INQ_ASSOC_MAX_COV) return cfail(INQ_ERR_ARG, "%s: %u covariates (at most %d)", fn, n_cov, INQ_ASSOC_MAX_COV);
    return INQ_OK;
}

// y: n_samples x n_traits row-major, NaN allowed (not used for that trait) when nan_ok; cov: finite
int assoc_check_values(const char *fn, int model, uint32_t n_samples, uint32_t n_traits, const double *y, bool nan_ok,
                       uint32_t n_cov, const double *cov)
{
    for (uint32_t s = 0; s < n_samples; ++s) {
        for (uint32_t t = 0; t < n_traits; ++t) {
            const double v = y[(size_t)s * n_traits + t];
            char what[32] = "trait";
            if (n_traits > 1 || nan_ok) snprintf(what, sizeof(what), "trait %u", t);
            if (nan_ok && std::isnan(v)) continue;
            if (!std::isfinite(v)) return cfail(INQ_ERR_ARG, "%s: %s of sample %u is not a finite number%s", fn, what, s, nan_ok ? " or NaN" : "");
            if (model != INQ_ASSOC_LINEAR && v != 0.0 && v != 1.0) return cfail(INQ_ERR_ARG, "%s: logistic %s of sample %u is not 0 or 1", fn, what, s);
        }
        for (uint32_t c = 0; c < n_cov; ++c)
            if (!std::isfinite(cov[(size_t)s * n_cov + c])) return cfail(INQ_ERR_ARG, "%s: covariate %u of sample %u is not a finite number", fn, c, s);
    }
    return INQ_OK;
}

// One single-trait problem with several right-hand sides: the traits of one sample set.
struct AssocGroup {
    std::vector<uint32_t> idx;                 // its samples (columns of the haplotype rows) in order; empty: all of them
    std::vector<uint32_t> traits;              // its traits (columns of y)
    std::vector<double> design, shift, y;      // prepared over its samples; y: traits.size() x samples
};

// The kernels' inputs over the group's samples: design rows [1, covariates centred by their mean, 0 (x), 0 ...] (row
// stride P), the P column shifts, and each trait (column t of y, row stride ld), centred by its mean for the linear model.
void assoc_prepare(AssocGroup &gr, int model, int P, uint32_t n_all, uint32_t n_cov, const double *cov, const double *y, uint32_t ld)
{
    const uint32_t n = gr.idx.empty() ? n_all : (uint32_t)gr.idx.size();
    auto sample = [&](uint32_t s) -> size_t { return gr.idx.empty() ? s : gr.idx[s]; };
    gr.design.assign((size_t)n * P, 0.0);
    gr.shift.assign(P, 0.0);
    for (uint32_t c = 0; c < n_cov; ++c) {
        double m = 0.0;
        for (uint32_t s = 0; s < n; ++s) m += cov[sample(s) * n_cov + c];
        gr.shift[1 + c] = m / n;
    }
    for (uint32_t s = 0; s < n; ++s) {
        gr.design[(size_t)s * P] = 1.0;
        for (uint32_t c = 0; c < n_cov; ++c) gr.design[(size_t)s * P + 1 + c] = cov[sample(s) * n_cov + c] - gr.shift[1 + c];
    }
    gr.y.resize(gr.traits.size() * (size_t)n);
    for (size_t j = 0; j < gr.traits.size(); ++j) {
        double *yj = gr.y.data() + j * n;
        for (uint32_t s = 0; s < n; ++s) yj[s] = y[sample(s) * ld + gr.traits[j]];
        if (model == INQ_ASSOC_LINEAR) {
            double m = 0.0;
            for (uint32_t s = 0; s < n; ++s) m += yj[s];
            m /= n;
            for (uint32_t s = 0; s < n; ++s) yj[s] -= m;
        }
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
    if (const int rc = assoc_check_args("inq_assoc", model, predictor, n_cov)) return rc;
    if (n_rows == 0) return INQ_OK;
    if (n_samples == 0) return cfail(INQ_ERR_ARG, "inq_assoc: no samples");
    if (!haps || !y || (n_cov && !cov) || !beta || !se || !stat || !p || !n_used || !status) return cfail(INQ_ERR_ARG, "inq_assoc: NULL array");
    if ((n_rows + kAWarps - 1) / kAWarps > 0x7FFFFFFFull) return cfail(INQ_ERR_TOO_LARGE, "inq_assoc: too many rows");
    if (const int rc = assoc_check_values("inq_assoc", model, n_samples, 1, y, false, n_cov, cov)) return rc;
    const uint32_t pdim = n_cov + 2;
    const int P = assoc_width(pdim);
    AssocGroup gr;
    gr.traits = {0};
    assoc_prepare(gr, model, P, n_samples, n_cov, cov, y, 1);

    CC_TRY(cudaSetDevice(device));
    Guard g;
    CC_TRY(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking));
    CC_TRY(cudaEventCreate(&g.e0));
    CC_TRY(cudaEventCreate(&g.e1));
    const size_t hap_bytes = (size_t)n_rows * 2 * n_samples * sizeof(double);
    void *d_haps, *d_des, *d_shift, *d_y, *d_res, *d_n, *d_st, *d_it;
    CC_TRY(g.alloc(&d_haps, hap_bytes));
    CC_TRY(g.alloc(&d_des, gr.design.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_shift, gr.shift.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_y, n_samples * sizeof(double)));
    CC_TRY(g.alloc(&d_res, (size_t)n_rows * 4 * sizeof(double)));
    CC_TRY(g.alloc(&d_n, (size_t)n_rows * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_st, (size_t)n_rows));
    CC_TRY(g.alloc(&d_it, (size_t)n_rows));
    CC_TRY(cudaMemcpyAsync(d_haps, haps, hap_bytes, cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_des, gr.design.data(), gr.design.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_shift, gr.shift.data(), gr.shift.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_y, gr.y.data(), n_samples * sizeof(double), cudaMemcpyHostToDevice, g.s));
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

int inq_assoc_traits(int device, int model, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
                     uint32_t n_traits, const double *y, uint32_t n_cov, const double *cov, double *beta, double *se,
                     double *stat, double *p, uint32_t *n_used, uint8_t *status, uint8_t *n_iter, float *ms_kernel)
{
    using namespace inqa;
    if (ms_kernel) *ms_kernel = 0.f;
    if (const int rc = assoc_check_args("inq_assoc_traits", model, predictor, n_cov)) return rc;
    if (n_traits == 0) return cfail(INQ_ERR_ARG, "inq_assoc_traits: no traits");
    if (n_rows == 0) return INQ_OK;
    if (n_samples == 0) return cfail(INQ_ERR_ARG, "inq_assoc_traits: no samples");
    if (!haps || !y || (n_cov && !cov) || !beta || !se || !stat || !p || !n_used || !status) return cfail(INQ_ERR_ARG, "inq_assoc_traits: NULL array");
    if (n_rows > (uint64_t)SIZE_MAX / 64 / n_traits) return cfail(INQ_ERR_TOO_LARGE, "inq_assoc_traits: %llu rows x %u traits", (unsigned long long)n_rows, n_traits);
    if (const int rc = assoc_check_values("inq_assoc_traits", model, n_samples, n_traits, y, true, n_cov, cov)) return rc;
    // group the traits by their sample set (NaN pattern), groups in the order of their first trait
    std::vector<AssocGroup> groups;
    {
        std::vector<std::vector<bool>> masks;
        for (uint32_t t = 0; t < n_traits; ++t) {
            std::vector<bool> m(n_samples);
            uint32_t cnt = 0;
            for (uint32_t s = 0; s < n_samples; ++s) cnt += m[s] = !std::isnan(y[(size_t)s * n_traits + t]);
            if (!cnt) return cfail(INQ_ERR_ARG, "inq_assoc_traits: trait %u has no value (every sample NaN)", t);
            size_t k = 0;
            while (k < masks.size() && masks[k] != m) ++k;
            if (k == masks.size()) {
                masks.push_back(m);
                groups.emplace_back();
                if (cnt < n_samples)
                    for (uint32_t s = 0; s < n_samples; ++s)
                        if (m[s]) groups[k].idx.push_back(s);
            }
            groups[k].traits.push_back(t);
        }
    }
    const uint32_t pdim = n_cov + 2;
    const int P = assoc_width(pdim);
    const int K = lin_traits_chunk(P);
    const uint64_t blocks = (n_rows + kAWarps - 1) / kAWarps;
    for (const AssocGroup &gr : groups) {
        const uint64_t per = model == INQ_ASSOC_LINEAR ? (gr.traits.size() + K - 1) / K : gr.traits.size();
        if (blocks > 0x7FFFFFFFull / per)
            return cfail(INQ_ERR_TOO_LARGE, "inq_assoc_traits: %llu rows x %zu traits of one sample set exceed the launch shape",
                         (unsigned long long)n_rows, gr.traits.size());
    }
    for (AssocGroup &gr : groups) assoc_prepare(gr, model, P, n_samples, n_cov, cov, y, n_traits);

    CC_TRY(cudaSetDevice(device));
    Guard g;
    CC_TRY(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking));
    CC_TRY(cudaEventCreate(&g.e0));
    CC_TRY(cudaEventCreate(&g.e1));
    // the haplotype matrix goes to the device once; each group reads its samples through its index
    const size_t hap_bytes = (size_t)n_rows * 2 * n_samples * sizeof(double), cells = (size_t)n_rows * n_traits;
    void *d_haps, *d_res, *d_n, *d_st, *d_it;
    CC_TRY(g.alloc(&d_haps, hap_bytes));
    CC_TRY(g.alloc(&d_res, cells * 4 * sizeof(double)));
    CC_TRY(g.alloc(&d_n, cells * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_st, cells));
    CC_TRY(g.alloc(&d_it, cells));
    CC_TRY(cudaMemcpyAsync(d_haps, haps, hap_bytes, cudaMemcpyHostToDevice, g.s));
    struct DevGroup { const double *des, *shift, *y; const uint32_t *idx, *tcol; };
    std::vector<DevGroup> dg(groups.size());
    auto upload = [&](const void *src, size_t bytes, const void **dst) -> int {
        void *q;
        CC_TRY(g.alloc(&q, bytes));
        CC_TRY(cudaMemcpyAsync(q, src, bytes, cudaMemcpyHostToDevice, g.s));
        *dst = q;
        return INQ_OK;
    };
    for (size_t k = 0; k < groups.size(); ++k) {
        const AssocGroup &gr = groups[k];
        DevGroup &d = dg[k];
        int rc = upload(gr.design.data(), gr.design.size() * sizeof(double), (const void **)&d.des);
        if (!rc) rc = upload(gr.shift.data(), gr.shift.size() * sizeof(double), (const void **)&d.shift);
        if (!rc) rc = upload(gr.y.data(), gr.y.size() * sizeof(double), (const void **)&d.y);
        if (!rc) rc = upload(gr.traits.data(), gr.traits.size() * sizeof(uint32_t), (const void **)&d.tcol);
        d.idx = nullptr;
        if (!rc && !gr.idx.empty()) rc = upload(gr.idx.data(), gr.idx.size() * sizeof(uint32_t), (const void **)&d.idx);
        if (rc) return rc;
    }
    double *r = (double *)d_res;
    const AssocOut out{r, r + cells, r + 2 * cells, r + 3 * cells, (uint32_t *)d_n, (uint8_t *)d_st, (uint8_t *)d_it};
    const int mx = predictor == INQ_ASSOC_MAX;
    const double *dh = (const double *)d_haps;
    CC_TRY(cudaEventRecord(g.e0, g.s));
    for (size_t k = 0; k < groups.size(); ++k) {
        const DevGroup &d = dg[k];
        const uint32_t ng = groups[k].idx.empty() ? n_samples : (uint32_t)groups[k].idx.size(), nt = (uint32_t)groups[k].traits.size();
        with_width(P, [&](auto width) {
            constexpr int W = decltype(width)::value;
            if (model == INQ_ASSOC_LINEAR) {
                constexpr int KW = lin_traits_chunk(W);
                const unsigned grid = (unsigned)(blocks * ((nt + KW - 1) / KW));
                k_assoc_linear_traits<W, KW><<<grid, kAWarps * 32, 0, g.s>>>(dh, n_rows, n_samples, d.idx, ng, pdim, mx, d.des, d.shift, d.y, nt,
                                                                            d.tcol, n_traits, out);
            } else {
                const unsigned grid = (unsigned)(blocks * nt);
                if (model == INQ_ASSOC_FIRTH)
                    k_assoc_traits<W, true><<<grid, kAWarps * 32, 0, g.s>>>(dh, n_rows, n_samples, d.idx, ng, pdim, mx, d.des, d.shift, d.y, nt, d.tcol, n_traits, out);
                else
                    k_assoc_traits<W, false><<<grid, kAWarps * 32, 0, g.s>>>(dh, n_rows, n_samples, d.idx, ng, pdim, mx, d.des, d.shift, d.y, nt, d.tcol, n_traits, out);
            }
        });
        CC_TRY(cudaGetLastError());
    }
    CC_TRY(cudaEventRecord(g.e1, g.s));
    CC_TRY(cudaMemcpyAsync(beta, r, cells * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(se, r + cells, cells * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(stat, r + 2 * cells, cells * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(p, r + 3 * cells, cells * sizeof(double), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(n_used, d_n, cells * sizeof(uint32_t), cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaMemcpyAsync(status, d_st, cells, cudaMemcpyDeviceToHost, g.s));
    if (n_iter) CC_TRY(cudaMemcpyAsync(n_iter, d_it, cells, cudaMemcpyDeviceToHost, g.s));
    CC_TRY(cudaStreamSynchronize(g.s));
    if (ms_kernel) cudaEventElapsedTime(ms_kernel, g.e0, g.e1);
    return INQ_OK;
}

int inq_assoc_cox(int device, int ties, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
                  const double *time, const uint8_t *event, uint32_t n_cov, const double *cov, double *beta, double *se,
                  double *stat, double *p, uint32_t *n_used, uint8_t *status, uint8_t *n_iter, float *ms_kernel)
{
    using namespace inqa;
    if (ms_kernel) *ms_kernel = 0.f;
    if (ties != INQ_COX_EFRON && ties != INQ_COX_BRESLOW) return cfail(INQ_ERR_ARG, "inq_assoc_cox: unknown ties method %d", ties);
    if (const int rc = assoc_check_args("inq_assoc_cox", INQ_ASSOC_LINEAR, predictor, n_cov)) return rc;
    if (n_rows == 0) return INQ_OK;
    if (n_samples == 0) return cfail(INQ_ERR_ARG, "inq_assoc_cox: no samples");
    if (!haps || !time || !event || (n_cov && !cov) || !beta || !se || !stat || !p || !n_used || !status) return cfail(INQ_ERR_ARG, "inq_assoc_cox: NULL array");
    if ((n_rows + kAWarps - 1) / kAWarps > 0x7FFFFFFFull) return cfail(INQ_ERR_TOO_LARGE, "inq_assoc_cox: too many rows");
    for (uint32_t s = 0; s < n_samples; ++s) {
        if (!std::isfinite(time[s])) return cfail(INQ_ERR_ARG, "inq_assoc_cox: time of sample %u is not a finite number", s);
        if (event[s] > 1) return cfail(INQ_ERR_ARG, "inq_assoc_cox: event of sample %u is not 0 or 1", s);
    }
    std::vector<double> ev(event, event + n_samples);
    if (const int rc = assoc_check_values("inq_assoc_cox", INQ_ASSOC_LINEAR, n_samples, 1, ev.data(), false, n_cov, cov)) return rc;
    // the samples in ascending time order (stable: ties keep the sample order), and the rank of each one's distinct time
    AssocGroup gr;
    gr.traits = {0};
    gr.idx.resize(n_samples);
    for (uint32_t s = 0; s < n_samples; ++s) gr.idx[s] = s;
    std::stable_sort(gr.idx.begin(), gr.idx.end(), [&](uint32_t a, uint32_t b) { return time[a] < time[b]; });
    std::vector<uint32_t> tg(n_samples);
    for (uint32_t s = 1; s < n_samples; ++s) tg[s] = tg[s - 1] + (time[gr.idx[s]] != time[gr.idx[s - 1]]);
    const uint32_t pdim = n_cov + 2;
    const int P = assoc_width(pdim);
    assoc_prepare(gr, INQ_ASSOC_LOGISTIC, P, n_samples, n_cov, cov, ev.data(), 1);      // y: the event, not centred

    CC_TRY(cudaSetDevice(device));
    Guard g;
    CC_TRY(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking));
    CC_TRY(cudaEventCreate(&g.e0));
    CC_TRY(cudaEventCreate(&g.e1));
    // grid-stride over blocks of loci: a grid of resident CTAs, its scratch (one entry per sample and warp) <= 1 GiB
    int sms = 0, per_sm = 0;
    CC_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CC_TRY(cox_occupancy(P, ties == INQ_COX_EFRON, &per_sm));
    const uint64_t blocks = (n_rows + kAWarps - 1) / kAWarps;
    const uint64_t slot_bytes = (uint64_t)kAWarps * n_samples * sizeof(double4);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min({blocks, (uint64_t)sms * std::max(per_sm, 1), (uint64_t)((1ull << 30) / slot_bytes)}));
    const size_t hap_bytes = (size_t)n_rows * 2 * n_samples * sizeof(double);
    void *d_haps, *d_des, *d_shift, *d_y, *d_idx, *d_tg, *d_scr, *d_res, *d_n, *d_st, *d_it;
    CC_TRY(g.alloc(&d_haps, hap_bytes));
    CC_TRY(g.alloc(&d_des, gr.design.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_shift, gr.shift.size() * sizeof(double)));
    CC_TRY(g.alloc(&d_y, n_samples * sizeof(double)));
    CC_TRY(g.alloc(&d_idx, n_samples * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_tg, n_samples * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_scr, grid * slot_bytes));
    CC_TRY(g.alloc(&d_res, (size_t)n_rows * 4 * sizeof(double)));
    CC_TRY(g.alloc(&d_n, (size_t)n_rows * sizeof(uint32_t)));
    CC_TRY(g.alloc(&d_st, (size_t)n_rows));
    CC_TRY(g.alloc(&d_it, (size_t)n_rows));
    CC_TRY(cudaMemcpyAsync(d_haps, haps, hap_bytes, cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_des, gr.design.data(), gr.design.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_shift, gr.shift.data(), gr.shift.size() * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_y, gr.y.data(), n_samples * sizeof(double), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_idx, gr.idx.data(), n_samples * sizeof(uint32_t), cudaMemcpyHostToDevice, g.s));
    CC_TRY(cudaMemcpyAsync(d_tg, tg.data(), n_samples * sizeof(uint32_t), cudaMemcpyHostToDevice, g.s));
    double *r = (double *)d_res;
    const AssocOut out{r, r + n_rows, r + 2 * n_rows, r + 3 * n_rows, (uint32_t *)d_n, (uint8_t *)d_st, (uint8_t *)d_it};
    const int mx = predictor == INQ_ASSOC_MAX;
    const double *dh = (const double *)d_haps, *dd = (const double *)d_des, *ds = (const double *)d_shift, *dy = (const double *)d_y;
    const uint32_t *di = (const uint32_t *)d_idx, *dt = (const uint32_t *)d_tg;
    double4 *dscr = (double4 *)d_scr;
    CC_TRY(cudaEventRecord(g.e0, g.s));
    cox_launch(P, ties == INQ_COX_EFRON, grid, g.s, dh, n_rows, n_samples, di, n_samples, pdim, mx, dd, ds, dy, dt, dscr, out);
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
