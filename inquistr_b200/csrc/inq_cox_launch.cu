// inq_cox_launch.cu -- the launches of k_assoc_cox (inq_assoc.cuh) for inq_assoc_cox (part of libinqcall.so).
// A translation unit of its own, so that the other assoc kernels in inq_cohort_capi.cu keep their compiled code.
#include "inq_assoc.cuh"

namespace inqa {

namespace {

// Calls f(kernel) with k_assoc_cox<P, efron> for the padded design width P: 4, 8, 16 or 32.
template <class F>
auto with_cox_kernel(int P, bool efron, F f)
{
    switch (P) {
    case 4: return efron ? f(k_assoc_cox<4, true>) : f(k_assoc_cox<4, false>);
    case 8: return efron ? f(k_assoc_cox<8, true>) : f(k_assoc_cox<8, false>);
    case 16: return efron ? f(k_assoc_cox<16, true>) : f(k_assoc_cox<16, false>);
    default: return efron ? f(k_assoc_cox<32, true>) : f(k_assoc_cox<32, false>);
    }
}

}  // namespace

cudaError_t cox_occupancy(int P, bool efron, int *per_sm)
{
    return with_cox_kernel(P, efron, [&](auto kernel) {
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kernel, kAWarps * 32, 0);
    });
}

void cox_launch(int P, bool efron, unsigned grid, cudaStream_t s, const double *haps, uint64_t n_rows, uint32_t n_all,
                const uint32_t *idx, uint32_t n_samples, uint32_t p, int use_max, const double *design, const double *shift,
                const double *event, const uint32_t *tgroup, double4 *scratch, AssocOut out)
{
    with_cox_kernel(P, efron, [&](auto kernel) {
        kernel<<<grid, kAWarps * 32, 0, s>>>(haps, n_rows, n_all, idx, n_samples, p, use_max, design, shift, event, tgroup,
                                             scratch, out);
        return 0;
    });
}

}  // namespace inqa
