// inq_assoc.cuh -- sm_100a kernels of `assoc`: per-locus regression of a trait on STR length. k_assoc fits the
// linear and the logistic model, k_assoc_firth the Firth-penalized logistic model (DESIGN.md 5e). For several traits
// (inq_assoc_traits), k_assoc_traits runs the same per-locus fits once per trait, and k_assoc_linear_traits shares one
// Gram matrix per locus between the linear traits of one sample set.
//
// All kernels have one layout. One warp per locus, four loci per CTA. The design is [1, covariates..., x] with x last
// (p <= 32 columns); lane j owns row j of the matrix being accumulated and entry j of the right-hand side, in f64
// registers (P = p rounded up to 4, 8, 16 or 32 is a template parameter, so the rows stay in registers). Each kernel
// keeps its own iteration logic and builds every sweep over the samples from the same routines:
//   locus_prepass    n (the samples with a call), the mean of x over them, and the sum of the trait over them.
//   stage_tile       the CTA stages a tile of 32 samples of the design rows shared by all loci (intercept +
//                    covariates, centred by their mean over the samples used) and of the trait in shared memory, so
//                    the sample count is not bounded by shared memory.
//   lane_x           lane l reads sample s0 + l of its locus (two haplotype values) and forms the centred predictor.
//   lane_eta         eta of that sample under the warp's coefficients; the kernel then forms the sample's weight W and
//                    the value v its right-hand side is built from.
//   accumulate_tile  the warp walks the valid samples of the tile (ballot) and every lane adds its row's terms of
//                    sum W u u' and of the right-hand side, and of the uncentred G_jj of the rank rule.
//   ldl_solve        symmetric Gaussian elimination (LDL') without pivoting, one row per lane, over the columns the
//                    caller keeps (a dropped column gets coefficient 0), then back substitution.
//   write_tail       NaN for the loci without a fit; n, status and the iteration count of every locus.
// The warps of a CTA run their sweeps in lock step (the tiles are shared); a warp whose locus is done idles.
//
// The predictor is centred per locus (mean over the samples used there), so the normal equations see centred
// columns. The rank rule compares each elimination pivot d_j (the weighted residual sum of squares of column j
// after the kept earlier columns, which centring does not change) with 1e-10 * G_jj of the UNcentred design.
// An aliased column is skipped (coefficient 0, rank - 1). With x last, (G^-1)_xx = 1 / d_x.
#pragma once

#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "../../include/inqcohort.h"

namespace inqa {

constexpr int kAWarps = 4;                 // loci per CTA
constexpr int kATile = 32;                 // samples per shared-memory tile
constexpr int kAMaxIter = 25;              // glm.control(maxit = 25)
constexpr double kAEpsilon = 1e-8;         // glm.control(epsilon = 1e-8)
constexpr double kAAlias = 1e-10;          // pivot d_j <= kAAlias * G_jj: column j aliased

// R's logit link (src/library/stats/src/family.c): THRESH = 30, MTHRESH = -30, INVEPS = 1 / DBL_EPSILON.
// linkinv gives mu = t / (1 + t) and also 1 - mu = 1 / (1 + t): R forms 1 - mu by subtraction, which keeps only
// eps / (1 - mu) of relative precision; for a misclassified sample near mu = 1 the IRLS term W (y - mu) / mu.eta is
// of order 1 and would inherit that error (1e-8 at |eta| = 18). Same model, no cancellation.
__host__ __device__ inline void logit_linkinv(double eta, double *mu, double *omu)
{
    const double t = eta < -30.0 ? DBL_EPSILON : (eta > 30.0 ? 1.0 / DBL_EPSILON : exp(eta));
    *mu = t / (1.0 + t);
    *omu = 1.0 / (1.0 + t);
}
__host__ __device__ inline double logit_mu_eta(double eta)
{
    const double opexp = 1.0 + exp(eta);
    return (eta > 30.0 || eta < -30.0) ? DBL_EPSILON : exp(eta) / (opexp * opexp);
}

// regularised incomplete beta I_x(a, b), continued fraction (modified Lentz), f64
__device__ inline double betacf(double a, double b, double x)
{
    const double tiny = 1e-300;
    double c = 1.0, d = 1.0 - (a + b) * x / (a + 1.0);
    if (fabs(d) < tiny) d = tiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= 1000; ++m) {
        const double m2 = 2.0 * m;
        double aa = m * (b - m) * x / ((a + m2 - 1.0) * (a + m2));
        d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d; h *= d * c;
        aa = -(a + m) * (a + b + m) * x / ((a + m2) * (a + m2 + 1.0));
        d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < 1e-16) break;
    }
    return h;
}
__device__ inline double betai(double a, double b, double x)
{
    if (x <= 0.0) return 0.0;
    if (x >= 1.0) return 1.0;
    const double lf = lgamma(a + b) - lgamma(a) - lgamma(b) + a * log(x) + b * log1p(-x);
    if (x < (a + 1.0) / (a + b + 2.0)) return exp(lf) * betacf(a, b, x) / a;
    return 1.0 - exp(lf) * betacf(b, a, 1.0 - x) / b;
}
// two-sided p of Student t with df degrees of freedom
__device__ inline double t_two_sided(double t, double df)
{
    if (t != t) return t;
    return betai(0.5 * df, 0.5, df / (df + t * t));
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct AssocOut {
    double *beta, *se, *stat, *p;
    uint32_t *n_used;
    uint8_t *status, *n_iter;
};

__device__ __forceinline__ double predictor(double2 v, int use_max) { return use_max ? fmax(v.x, v.y) : v.x + v.y; }

// The samples of one trait group (k_assoc_traits, k_assoc_linear_traits): sample s of the group is column idx[s] of
// the locus's haplotype row, or column s when idx is null (the group has every sample of the row).
struct SampleSubset {
    const double2 *h;
    const uint32_t *__restrict__ idx;
    __device__ __forceinline__ double2 operator[](uint32_t s) const { return idx ? h[idx[s]] : h[s]; }
};

struct LocusSums {
    uint32_t n;                            // samples with a call
    double xbar, cases;                    // mean of x over them, sum of the trait over them
};

// H: the locus's haplotype pairs, h[s] for sample s: a double2 pointer, or SampleSubset
template <class H>
__device__ __forceinline__ LocusSums locus_prepass(const H &h, const double *__restrict__ y, uint32_t n_samples,
                                                   int use_max, bool have, uint32_t lane)
{
    double sx = 0.0, sy = 0.0;
    uint32_t cnt = 0;
    if (have)
        for (uint32_t s = lane; s < n_samples; s += 32) {
            const double x = predictor(h[s], use_max);
            if (x == x) { sx += x; sy += y[s]; ++cnt; }
        }
    uint32_t n = cnt;
#pragma unroll
    for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    return {n, n ? warp_sum(sx) / n : 0.0, warp_sum(sy)};
}

// design: n_samples x P (row stride P): [1, centred covariates..., 0 (the slot of x), 0 padding]
// s_des has the odd row stride P + 1 in doubles, so lane-per-row reads spread over the banks. tid is threadIdx.x of the
// caller: the kernel's read carries the range [0, kAWarps * 32) of __launch_bounds__, and with it the compiler needs no
// guard in front of the first trip of the loop below (a read here would get a guard branch per tile).
// K traits (k_assoc_linear_traits): s_y holds kATile rows of YS doubles, trait k of sample r at s_y[r * YS + k] (0 for
// k >= kn), read from y[k * n_samples + s].
template <int P, int K = 1, int YS = 1>
__device__ __forceinline__ void stage_tile(double (*s_des)[P + 1], double *s_y, const double *__restrict__ design,
                                           const double *__restrict__ y, uint32_t s0, uint32_t n_samples, uint32_t tid,
                                           uint32_t kn = 1)
{
    __syncthreads();
    for (uint32_t t = tid; t < (uint32_t)kATile * P; t += blockDim.x) {
        const uint32_t r = t / P, c = t % P, s = s0 + r;
        s_des[r][c] = s < n_samples ? design[(uint64_t)s * P + c] : 0.0;
    }
    if (tid < kATile)
#pragma unroll
        for (int k = 0; k < K; ++k)
            s_y[tid * YS + k] = s0 + tid < n_samples && (uint32_t)k < kn ? y[(uint64_t)k * n_samples + (s0 + tid)] : 0.0;
    __syncthreads();
}

// x - xbar of sample s; NaN for a sample without a call and for the padding of the last tile
template <class H>
__device__ __forceinline__ double lane_x(const H &h, uint32_t s, uint32_t n_samples, int use_max, double xbar)
{
    double xt = __longlong_as_double(0x7ff8000000000000ll);
    if (s < n_samples) xt = predictor(h[s], use_max) - xbar;
    return xt;
}

template <int P>
__device__ __forceinline__ double lane_eta(const double *beta, const double *des, uint32_t xcol, double xt)
{
    double eta = 0.0;
#pragma unroll
    for (int k = 0; k < P; ++k) eta = fma(beta[k], des[k], eta);
    return fma(beta[xcol], xt, eta);       // the x slot of s_des is 0
}

// The ballot walk over the valid samples of the tile: u = [design row, x] of sample i, lane j adds W_i u_i u_ij to
// row j of G (its x entry to gx: a run-time index into G would put G in local memory; put_x moves it in),
// rhs_term(rhs, W_i u_ij, u_ij, v_i, i) adds its terms to rhs and, with with_diag, W_i (u_ij + shift_j)^2 to diag,
// the uncentred G_jj. Each kernel keeps its own expression for the right-hand side: fma(W u, z, .) and fma(W z, u, .)
// round differently; k_assoc_linear_traits reads its K values of sample i from shared memory (v unused).
template <int P, class Rhs, class RhsTerm>
__device__ __forceinline__ void accumulate_tile(double (&G)[P], double &gx, Rhs &rhs, double &diag,
                                                const double (*s_des)[P + 1], uint32_t lane, uint32_t xcol, bool valid,
                                                double xt, double W, double v, double my_shift, bool with_diag,
                                                RhsTerm rhs_term)
{
    unsigned m = __ballot_sync(0xffffffffu, valid);
    while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        const double xi = __shfl_sync(0xffffffffu, xt, i);
        const double wi = __shfl_sync(0xffffffffu, W, i);
        const double vi = __shfl_sync(0xffffffffu, v, i);
        const double uj = lane == xcol ? xi : (lane < P ? s_des[i][lane < P ? lane : 0] : 0.0);
        const double a = wi * uj;
#pragma unroll
        for (int k = 0; k < P; ++k) G[k] = fma(a, s_des[i][k], G[k]);
        gx = fma(a, xi, gx);
        rhs_term(rhs, a, uj, vi, i);
        if (with_diag) {
            const double raw = uj + my_shift;
            diag = fma(wi * raw, raw, diag);
        }
    }
}

template <int P>
__device__ __forceinline__ void put_x(double (&G)[P], double gx, uint32_t xcol)
{
#pragma unroll
    for (int k = 0; k < P; ++k) if (k == (int)xcol) G[k] = gx;
}

// Solves G b_r = rhs_r for R right-hand sides over the columns c < p that keep(c, d_c) accepts, d_c the pivot of column
// c after the kept earlier columns; G is eliminated once and every right-hand side sees the operations of a solve of
// its own. G and rhs are overwritten. -> b: this lane's coefficients (0 for a dropped column and for lanes >= p).
template <int P, int R, class Keep>
__device__ __forceinline__ void ldl_solve(double (&G)[P], double (&rhs)[R], double (&b)[R], uint32_t p, uint32_t lane,
                                          Keep keep)
{
    uint32_t kept = 0;
#pragma unroll
    for (int c = 0; c < P; ++c) {
        if (c >= (int)p) break;
        const double d = __shfl_sync(0xffffffffu, G[c], c);
        if (!keep(c, d)) continue;
        kept |= 1u << c;
        const double l = G[c] / d;
        double bc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) bc[r] = __shfl_sync(0xffffffffu, rhs[r], c);
#pragma unroll
        for (int k = c + 1; k < P; ++k) {
            if (k >= (int)p) break;
            const double gck = __shfl_sync(0xffffffffu, G[k], c);
            if ((int)lane > c) G[k] = fma(-l, gck, G[k]);
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if ((int)lane > c) rhs[r] = fma(-l, bc[r], rhs[r]);
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        double acc = 0.0, br = 0.0;
#pragma unroll
        for (int c = P - 1; c >= 0; --c) {
            if (c >= (int)p || !((kept >> c) & 1u)) continue;
            const double bc = __shfl_sync(0xffffffffu, (rhs[r] - acc) / G[c], c);
            if ((int)lane == c) br = bc;
            if ((int)lane < c) acc = fma(G[c], bc, acc);
        }
        b[r] = br;
    }
}

template <int P>
__device__ __forceinline__ void publish_beta(double *s_beta, uint32_t lane, double b)
{
    __syncwarp();
    if (lane < P) s_beta[lane] = b;
    __syncwarp();
}

__device__ __forceinline__ void write_tail(const AssocOut &out, uint64_t row, bool have, uint32_t lane, uint32_t n,
                                           uint8_t status, int n_iter)
{
    if (have && lane == 0) {
        if (status == INQ_ASSOC_FEW_SAMPLES || status == INQ_ASSOC_SINGULAR) {
            const double nan = __longlong_as_double(0x7ff8000000000000ll);
            out.beta[row] = nan; out.se[row] = nan; out.stat[row] = nan; out.p[row] = nan;
        }
        out.n_used[row] = n;
        out.status[row] = status;
        if (out.n_iter) out.n_iter[row] = (uint8_t)n_iter;
    }
}

// Linear: pass 0 accumulates G (W = 1, z = y - mean y), solve, pass 1 sums the squared residuals.
// Logistic (R's glm.fit without step-halving): pass t evaluates eta = X beta_t (t = 0: the start mu = (y + 1/2) / 2),
// mu, the deviance of beta_t, and the weights / working response of the next solve, and accumulates that solve's G.
// shift: P column shifts (covariate means; 0 for the intercept and x), to rebuild the uncentred G_jj
// y    : n_samples trait values (linear: centred by their mean)
// One locus of k_assoc / k_assoc_traits: h its haplotype pairs, have = the warp has a locus, row its output index.
template <int P, class H>
__device__ __forceinline__ void assoc_fit(uint32_t tid, const H &h, bool have, uint64_t row, uint32_t n_samples, uint32_t p, int logistic,
                                          int use_max, const double *__restrict__ design, const double *__restrict__ shift,
                                          const double *__restrict__ y, const AssocOut &out)
{
    __shared__ double s_des[kATile][P + 1];
    __shared__ double s_y[kATile];
    __shared__ double s_beta[kAWarps][P];
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const uint32_t xcol = p - 1;
    const auto [n, xbar, cases] = locus_prepass(h, y, n_samples, use_max, have, lane);

    uint8_t status = INQ_ASSOC_OK;
    bool done = !have;
    if (have && (n == 0 || (logistic && (cases == 0.0 || cases == (double)n)))) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
    if (lane < P) s_beta[warp][lane] = 0.0;

    const double my_shift = lane == xcol ? xbar : (lane < P ? shift[lane] : 0.0);
    double beta_lane = 0.0, dx = 0.0, dev_old = 0.0;
    int iter = 0, pass = 0, rank = 0;
    for (;;) {
        if (__syncthreads_and(done)) break;
        // per-pass accumulators: row `lane` of G, X'Wz, uncentred G_jj; deviance / RSS and the separation test
        double G[P];
#pragma unroll
        for (int k = 0; k < P; ++k) G[k] = 0.0;
        double gx = 0.0, rhs = 0.0, diag = 0.0;
        double dsum = 0.0;
        bool sep_l = false;
        const bool need_gram = !done && (logistic || pass == 0);
        for (uint32_t s0 = 0; s0 < n_samples; s0 += kATile) {
            stage_tile<P>(s_des, s_y, design, y, s0, n_samples, tid);
            if (done) continue;
            const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
            const bool valid = xt == xt;
            const double yl = s_y[lane];
            double eta = lane_eta<P>(s_beta[warp], s_des[lane], xcol, xt);
            double W = 1.0, z = yl;
            if (logistic) {
                if (pass == 0) {
                    const double mu0 = (yl + 0.5) * 0.5;
                    eta = log(mu0 / (1.0 - mu0));
                }
                double mu, omu;
                logit_linkinv(eta, &mu, &omu);
                const double me = logit_mu_eta(eta);
                if (valid) {
                    dsum += yl != 0.0 ? -2.0 * log(mu) : -2.0 * log(omu);
                    sep_l |= mu < 10.0 * DBL_EPSILON || omu < 10.0 * DBL_EPSILON;
                }
                W = me * me / (mu * omu);
                z = eta + (yl != 0.0 ? omu : -mu) / me;
            } else if (pass == 1 && valid) {
                const double r = yl - eta;
                dsum = fma(r, r, dsum);
            }
            if (!need_gram) continue;
            accumulate_tile<P>(G, gx, rhs, diag, s_des, lane, xcol, valid, xt, W, z, my_shift, true,
                               [](double &rhs, double a, double, double zi, int) { rhs = fma(a, zi, rhs); });
        }
        if (!done) {
            const double dev = warp_sum(dsum);             // deviance of the current coefficients (linear: RSS)
            const bool any_sep = __any_sync(0xffffffffu, sep_l);
            bool solve = true;
            if (!logistic && pass == 1) {
                // RSS known: t statistic
                const double df = (double)n - rank;
                const double sigma2 = dev / df;
                const double se = sqrt(sigma2 / dx);
                const double beta = __shfl_sync(0xffffffffu, beta_lane, xcol);
                if (lane == 0) {
                    const double t = beta / se;
                    out.beta[row] = beta; out.se[row] = se; out.stat[row] = t; out.p[row] = t_two_sided(t, df);
                }
                done = true;
                solve = false;
            } else if (logistic && pass > 0) {
                const double crit = fabs(dev - dev_old) / (fabs(dev) + 0.1);
                if (crit < kAEpsilon || iter == kAMaxIter) {
                    if (crit >= kAEpsilon) status = INQ_ASSOC_NO_CONVERGENCE;
                    else if (any_sep) status = INQ_ASSOC_SEPARATION;
                    const double se = sqrt(1.0 / dx);
                    const double beta = __shfl_sync(0xffffffffu, beta_lane, xcol);
                    if (lane == 0) {
                        const double zs = beta / se;
                        out.beta[row] = beta; out.se[row] = se; out.stat[row] = zs; out.p[row] = erfc(fabs(zs) * M_SQRT1_2);
                    }
                    done = true;
                    solve = false;
                }
            }
            dev_old = dev;
            if (solve) {
                put_x(G, gx, xcol);
                uint32_t kept = 0;
                double d_x = 0.0;
                double b[1], r1[1] = {rhs};
                ldl_solve<P>(G, r1, b, p, lane, [&](int c, double d) {
                    if (!(d > kAAlias * __shfl_sync(0xffffffffu, diag, c))) return false;   // aliased (or empty) column
                    kept |= 1u << c;
                    if (c == (int)xcol) d_x = d;
                    return true;
                });
                const int rk = __popc(kept);
                if (pass == 0) rank = rk;
                if (pass == 0 && n <= (uint32_t)rk) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
                else if (!((kept >> xcol) & 1u)) { status = INQ_ASSOC_SINGULAR; done = true; }
                else {
                    rank = rk;
                    dx = d_x;
                    beta_lane = b[0];
                    publish_beta<P>(s_beta[warp], lane, b[0]);
                    if (logistic) ++iter;
                }
            }
        }
        ++pass;
    }
    write_tail(out, row, have, lane, n, status, iter);
}

template <int P>
__global__ void __launch_bounds__(kAWarps * 32)
k_assoc(const double *__restrict__ haps, uint64_t n_rows, uint32_t n_samples, uint32_t p, int logistic, int use_max,
        const double *__restrict__ design, const double *__restrict__ shift, const double *__restrict__ y, AssocOut out)
{
    const uint32_t tid = threadIdx.x;
    const uint64_t row = (uint64_t)blockIdx.x * kAWarps + (tid >> 5);
    const bool have = row < n_rows;
    assoc_fit<P>(tid, reinterpret_cast<const double2 *>(haps + (have ? row : 0) * 2ull * n_samples), have, row, n_samples, p,
                 logistic, use_max, design, shift, y, out);
}

// ---------------------------------------------------------------------------------------------------------------
// Firth-penalized logistic regression (DESIGN.md 5e, Firth). Per locus two fits, the full one (free set F = K) and
// the null one (F = K \ {x}, beta_x = 0), each from beta = 0; K is the rank set decided at the first evaluation.
// A step is two sweeps over the samples:
//   A: at beta, eta, mu, w = mu (1 - mu), the deviance and I = X_K' W X_K; factor I = L D L' over K;
//      D* = deviance - log det I. If D* rose, beta moves half way back to beta_prev and A runs again (<= 5 times).
//   B: at the same beta, h_i = w_i x_i' I^-1 x_i, U* = X'(y - mu + h (1/2 - mu)), H = X' diag(w (1 + h)) X;
//      delta_F = H_FF^-1 U*_F, lambda^2 = delta_F . U*_F; converged below 1e-10, else beta += delta.
// For B, the factor of I is kept in per-warp shared memory as L^-1 (unit lower triangular) and 1/d, so lane l gets
// h of its own sample as w sum_c (1/d_c) ((L^-1 u)_c)^2 from dot products of broadcast rows of L^-1 with its design
// row u: no per-lane vector is held next to the accumulators. Centring x and the covariates is a unit-triangular
// change of columns; it leaves every quantity of the iteration, and log det I, unchanged.
constexpr int kFMaxSteps = 100;            // steps per fit
constexpr int kFMaxHalvings = 5;           // halvings per step
constexpr double kFLambda2 = 1e-10;        // convergence: delta_F . U*_F below this
constexpr double kFRise = 1e-12;           // halve when D* > D*_prev + kFRise (|D*_prev| + 1)

template <int P, class H>
__device__ __forceinline__ void firth_fit(uint32_t tid, const H &h, bool have, uint64_t row, uint32_t n_samples, uint32_t p, int use_max,
                                          const double *__restrict__ design, const double *__restrict__ shift,
                                          const double *__restrict__ y, const AssocOut &out)
{
    __shared__ double s_des[kATile][P + 1];
    __shared__ double s_y[kATile];
    __shared__ double s_beta[kAWarps][P];
    __shared__ double s_li[kAWarps][P][P];     // L^-1 of the warp's last factor of I (identity outside K)
    __shared__ double s_dinv[kAWarps][P];      // 1 / d_c for c in K, 0 elsewhere
    __shared__ double s_full[kAWarps][3];      // the full fit's beta_x, se and D*
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const uint32_t xcol = p - 1;
    const auto [n, xbar, cases] = locus_prepass(h, y, n_samples, use_max, have, lane);

    uint8_t status = INQ_ASSOC_OK;
    bool done = !have;
    if (have && (n == 0 || cases == 0.0 || cases == (double)n)) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
    if (lane < P) s_beta[warp][lane] = 0.0;

    const double my_shift = lane == xcol ? xbar : (lane < P ? shift[lane] : 0.0);
    // b / b_prev: this lane's coefficient (lane < P); dpen: D* at b; dpen_prev: D* at b_prev; dx: pivot of x in I
    double b = 0.0, b_prev = 0.0, dpen = 0.0, dpen_prev = 0.0, dx = 0.0;
    uint32_t kmask = 0;
    int fit = 0, t = 0, halvings = 0, t_full = 0;
    bool first = true, sweep_b = false, conv_full = false;
    for (;;) {
        if (__syncthreads_and(done)) break;
        // A: row `lane` of I, the deviance, the uncentred G_jj (first sweep only, for the rank rule)
        // B: row `lane` of H and U*_lane
        double G[P];
#pragma unroll
        for (int k = 0; k < P; ++k) G[k] = 0.0;
        double gx = 0.0, rhs = 0.0, diag = 0.0;
        double dsum = 0.0;
        for (uint32_t s0 = 0; s0 < n_samples; s0 += kATile) {
            stage_tile<P>(s_des, s_y, design, y, s0, n_samples, tid);
            if (done) continue;
            const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
            const bool valid = xt == xt;
            const double yl = s_y[lane];
            const double eta = lane_eta<P>(s_beta[warp], s_des[lane], xcol, xt);
            double mu, omu;
            logit_linkinv(eta, &mu, &omu);
            const double w = mu * omu;
            double W = w, r = 0.0;
            if (!sweep_b) {
                if (valid) dsum += yl != 0.0 ? -2.0 * log(mu) : -2.0 * log(omu);
            } else {
                // x' I^-1 x of this lane's sample: sum_c (1/d_c) z_c^2, z = L^-1 u, u = [design row, x]
                double q = 0.0;
#pragma unroll 1
                for (int c = 0; c < (int)p; ++c) {
                    double z = 0.0;
#pragma unroll 4
                    for (int k = 0; k <= c; ++k) z = fma(s_li[warp][k][c], s_des[lane][k], z);
                    if (c == (int)xcol) z = fma(s_li[warp][c][c], xt, z);
                    q = fma(s_dinv[warp][c] * z, z, q);
                }
                const double hh = w * q;
                W = w * (1.0 + hh);
                r = (yl != 0.0 ? omu : -mu) + hh * (0.5 - mu);
            }
            accumulate_tile<P>(G, gx, rhs, diag, s_des, lane, xcol, valid, xt, W, r, my_shift, first,
                               [](double &rhs, double, double uj, double ri, int) { rhs = fma(ri, uj, rhs); });
        }
        if (done) { continue; }
        put_x(G, gx, xcol);
        if (!sweep_b) {
            // LDL' of I over K (the first time: K by the rank rule); lane j > c keeps L_jc in G[c]
            const double dev = warp_sum(dsum);
            uint32_t kept = 0;
            double logdet = 0.0, d_x = 0.0, my_dinv = 0.0;
#pragma unroll
            for (int c = 0; c < P; ++c) {
                if (c >= (int)p) break;
                const double d = __shfl_sync(0xffffffffu, G[c], c);
                if (first) {
                    const double sc = __shfl_sync(0xffffffffu, diag, c);
                    if (!(d > kAAlias * sc)) continue;
                } else if (!((kmask >> c) & 1u)) continue;
                kept |= 1u << c;
                logdet += log(d);
                if (c == (int)xcol) d_x = d;
                if ((int)lane == c) my_dinv = 1.0 / d;
                const double l = G[c] / d;
#pragma unroll
                for (int k = c + 1; k < P; ++k) {
                    if (k >= (int)p) break;
                    const double gck = __shfl_sync(0xffffffffu, G[k], c);
                    if ((int)lane > c) G[k] = fma(-l, gck, G[k]);
                }
                if ((int)lane > c) G[c] = l;
            }
            if (first) {
                first = false;
                kmask = kept;
                if (n <= (uint32_t)__popc(kept)) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
                else if (!((kept >> xcol) & 1u)) { status = INQ_ASSOC_SINGULAR; done = true; }
                if (done) continue;
            }
            const double dnew = dev - logdet;
            if (t > 0 && dnew > dpen_prev + kFRise * (fabs(dpen_prev) + 1.0) && halvings < kFMaxHalvings) {
                b = 0.5 * (b + b_prev);
                ++halvings;
                publish_beta<P>(s_beta[warp], lane, b);
                continue;
            }
            dpen = dnew;
            dx = d_x;
            // L^-1 column by column from the rows of L in G (strictly lower, 0 outside K):
            // (L^-1)_jk = -sum_{m = k..j-1} L_jm (L^-1)_mk, lane j gets row j once rows k..j-1 are final.
            // Stored transposed, s_li[k][j] = (L^-1)_jk, so the lanes write consecutive words.
            const bool my_kept = (kmask >> lane) & 1u;
#pragma unroll
            for (int m = 0; m < P; ++m)
                if (!(m < (int)lane && my_kept && ((kmask >> m) & 1u))) G[m] = 0.0;
            __syncwarp();
#pragma unroll
            for (int k = 0; k < P; ++k) {
                double lk = (int)lane == k ? 1.0 : 0.0, acc = 0.0;
#pragma unroll
                for (int m = k; m < P - 1; ++m) {
                    const double v = __shfl_sync(0xffffffffu, lk, m);
                    acc = fma(G[m], v, acc);                  // G[m] = 0 unless m < lane
                    if ((int)lane == m + 1) lk = -acc;
                }
                if (lane < P) s_li[warp][k][lane] = lk;
            }
            if (lane < P) s_dinv[warp][lane] = my_dinv;
            __syncwarp();
            sweep_b = true;
            continue;
        }
        // B: delta_F = H_FF^-1 U*_F over F; rhs keeps U*
        sweep_b = false;
        const uint32_t fmask = fit == 0 ? kmask : kmask & ~(1u << xcol);
        double dl[1], r1[1] = {rhs};
        ldl_solve<P>(G, r1, dl, p, lane, [&](int c, double) { return ((fmask >> c) & 1u) != 0; });
        const double delta = dl[0];
        const double lam2 = warp_sum(lane < P && ((fmask >> lane) & 1u) ? delta * rhs : 0.0);
        const bool conv = lam2 < kFLambda2;
        if (!conv && t < kFMaxSteps) {
            b_prev = b;
            dpen_prev = dpen;
            b += delta;
            ++t;
            halvings = 0;
        } else if (fit == 0) {
            // full fit done: keep its result, start the null fit from beta = 0
            if (lane == xcol) { s_full[warp][0] = b; s_full[warp][1] = sqrt(1.0 / dx); s_full[warp][2] = dpen; }
            t_full = t;
            conv_full = conv;
            fit = 1;
            b = b_prev = 0.0;
            t = halvings = 0;
        } else {
            if (lane == 0) {
                const double stat = fmax(0.0, dpen - s_full[warp][2]);
                out.beta[row] = s_full[warp][0]; out.se[row] = s_full[warp][1]; out.stat[row] = stat; out.p[row] = erfc(sqrt(0.5 * stat));
            }
            if (!conv_full || !conv) status = INQ_ASSOC_NO_CONVERGENCE;
            done = true;
        }
        publish_beta<P>(s_beta[warp], lane, b);
    }
    write_tail(out, row, have, lane, n, status, t_full);
}

template <int P>
__global__ void __launch_bounds__(kAWarps * 32)
k_assoc_firth(const double *__restrict__ haps, uint64_t n_rows, uint32_t n_samples, uint32_t p, int use_max,
              const double *__restrict__ design, const double *__restrict__ shift, const double *__restrict__ y, AssocOut out)
{
    const uint32_t tid = threadIdx.x;
    const uint64_t row = (uint64_t)blockIdx.x * kAWarps + (tid >> 5);
    const bool have = row < n_rows;
    firth_fit<P>(tid, reinterpret_cast<const double2 *>(haps + (have ? row : 0) * 2ull * n_samples), have, row, n_samples, p,
                 use_max, design, shift, y, out);
}

// ---------------------------------------------------------------------------------------------------------------
// Several traits (inq_assoc_traits, DESIGN.md 5e, Several traits). A group is the traits of one sample set: its n_samples
// samples are columns idx[s] of the haplotype rows (stride n_all samples; idx null: all of them), and its design, shifts
// and traits (y: n_tr x n_samples, trait j of the group is output column tcol[j] of n_traits) are prepared over them
// exactly as inq_assoc prepares a single trait, so every trait's fit is the single-trait fit bit for bit.

// Logistic and Firth: W depends on the trait, so each CTA fits one trait of the group on kAWarps loci. The CTAs of one
// block of loci for all traits of the group are adjacent: the haplotype rows come from HBM once, the other traits hit L2.
template <int P, bool kFirth>
__global__ void __launch_bounds__(kAWarps * 32)
k_assoc_traits(const double *__restrict__ haps, uint64_t n_rows, uint32_t n_all, const uint32_t *__restrict__ idx,
               uint32_t n_samples, uint32_t p, int use_max, const double *__restrict__ design,
               const double *__restrict__ shift, const double *__restrict__ y, uint32_t n_tr,
               const uint32_t *__restrict__ tcol, uint32_t n_traits, AssocOut out)
{
    const uint32_t tid = threadIdx.x, j = blockIdx.x % n_tr;
    const uint64_t row = (uint64_t)(blockIdx.x / n_tr) * kAWarps + (tid >> 5);
    const bool have = row < n_rows;
    const SampleSubset h{reinterpret_cast<const double2 *>(haps + (have ? row : 0) * 2ull * n_all), idx};
    const uint64_t orow = row * n_traits + tcol[j];
    const double *yj = y + (uint64_t)j * n_samples;
    if constexpr (kFirth) firth_fit<P>(tid, h, have, orow, n_samples, p, use_max, design, shift, yj, out);
    else assoc_fit<P>(tid, h, have, orow, n_samples, p, 1, use_max, design, shift, yj, out);
}

// Linear, shared Gram: G = X'X and the rank rule depend on the samples and covariates only. Each CTA takes kAWarps loci
// and a chunk of up to K traits of the group (chunks of one block of loci adjacent, as above). Pass 0 accumulates G and
// the uncentred G_jj once and X'y of the K traits with the operations of k_assoc's pass 0; one elimination of G solves
// all K right-hand sides; pass 1 sums every trait's squared residuals. n, rank and the status are shared by the chunk.
// K, the traits of one chunk, for the padded width P: the most for which ptxas reports no spill and no stack frame
constexpr int lin_traits_chunk(int P) { return P <= 8 ? 16 : P == 16 ? 7 : 4; }

template <int P, int K>
__global__ void __launch_bounds__(kAWarps * 32)
k_assoc_linear_traits(const double *__restrict__ haps, uint64_t n_rows, uint32_t n_all, const uint32_t *__restrict__ idx,
                      uint32_t n_samples, uint32_t p, int use_max, const double *__restrict__ design,
                      const double *__restrict__ shift, const double *__restrict__ y, uint32_t n_tr,
                      const uint32_t *__restrict__ tcol, uint32_t n_traits, AssocOut out)
{
    constexpr int YS = K | 1;                  // odd row stride: lane-per-row reads of s_y spread over the banks
    __shared__ double s_des[kATile][P + 1];
    __shared__ double s_y[kATile * YS];
    __shared__ double s_beta[kAWarps][K][P];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t n_chunks = (n_tr + K - 1) / K, chunk = blockIdx.x % n_chunks, k0 = chunk * K;
    const uint32_t kn = min((uint32_t)K, n_tr - k0);
    const uint64_t row = (uint64_t)(blockIdx.x / n_chunks) * kAWarps + warp;
    const bool have = row < n_rows;
    const SampleSubset h{reinterpret_cast<const double2 *>(haps + (have ? row : 0) * 2ull * n_all), idx};
    const double *yk = y + (uint64_t)k0 * n_samples;
    const uint32_t xcol = p - 1;
    const auto [n, xbar, cases] = locus_prepass(h, yk, n_samples, use_max, have, lane);
    (void)cases;

    uint8_t status = INQ_ASSOC_OK;
    bool done = !have;
    if (have && n == 0) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
    const double my_shift = lane == xcol ? xbar : (lane < P ? shift[lane] : 0.0);

    // pass 0: row `lane` of G, X'y of each trait, uncentred G_jj
    double G[P];
#pragma unroll
    for (int k = 0; k < P; ++k) G[k] = 0.0;
    double gx = 0.0, rhs[K], diag = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) rhs[k] = 0.0;
    for (uint32_t s0 = 0; s0 < n_samples; s0 += kATile) {
        stage_tile<P, K, YS>(s_des, s_y, design, yk, s0, n_samples, tid, kn);
        if (done) continue;
        const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
        accumulate_tile<P>(G, gx, rhs, diag, s_des, lane, xcol, xt == xt, xt, 1.0, 0.0, my_shift, true,
                           [&](double (&r)[K], double a, double, double, int i) {
#pragma unroll
                               for (int k = 0; k < K; ++k) r[k] = fma(a, s_y[i * YS + k], r[k]);
                           });
    }
    int rank = 0;
    double dx = 0.0, b[K];
    if (!done) {
        put_x(G, gx, xcol);
        uint32_t kept = 0;
        ldl_solve<P>(G, rhs, b, p, lane, [&](int c, double d) {
            if (!(d > kAAlias * __shfl_sync(0xffffffffu, diag, c))) return false;   // aliased (or empty) column
            kept |= 1u << c;
            if (c == (int)xcol) dx = d;
            return true;
        });
        rank = __popc(kept);
        if (n <= (uint32_t)rank) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
        else if (!((kept >> xcol) & 1u)) { status = INQ_ASSOC_SINGULAR; done = true; }
        else {
            __syncwarp();
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (lane < P) s_beta[warp][k][lane] = b[k];
            __syncwarp();
        }
    }

    // pass 1: residual sum of squares of each trait
    double dsum[K];
#pragma unroll
    for (int k = 0; k < K; ++k) dsum[k] = 0.0;
    if (!__syncthreads_and(done))
        for (uint32_t s0 = 0; s0 < n_samples; s0 += kATile) {
            stage_tile<P, K, YS>(s_des, s_y, design, yk, s0, n_samples, tid, kn);
            if (done) continue;
            const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
            if (xt != xt) continue;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if ((uint32_t)k >= kn) break;
                const double r = s_y[lane * YS + k] - lane_eta<P>(s_beta[warp][k], s_des[lane], xcol, xt);
                dsum[k] = fma(r, r, dsum[k]);
            }
        }
    const double df = (double)n - rank;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if ((uint32_t)k >= kn) break;
        const uint64_t orow = row * n_traits + tcol[k0 + k];
        if (!done) {
            // as k_assoc's pass 1: the t statistic from the RSS
            const double dev = warp_sum(dsum[k]);
            const double se = sqrt(dev / df / dx);
            const double beta = __shfl_sync(0xffffffffu, b[k], xcol);
            if (lane == 0) {
                const double t = beta / se;
                out.beta[orow] = beta; out.se[orow] = se; out.stat[orow] = t; out.p[orow] = t_two_sided(t, df);
            }
        }
        write_tail(out, orow, have, lane, n, status, 0);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Cox proportional hazards (inq_assoc_cox, DESIGN.md 5e, Cox): partial likelihood of (time, event) on u = [covariates...,
// x] (no intercept: column 0 of the shared design never enters the kept set K), Efron or Breslow ties, Newton
// iteration with coxph.fit's control flow. The samples come in ascending time order (idx), event[s] is 0 or 1 and
// tgroup[s] the rank of sample s's distinct time. One evaluation at beta is two sweeps over the samples:
//   A  descending time, tiles last to first, lanes 31 to 0: the risk-set sums B (samples of R(tau) outside D(tau)) and
//      the pending tie group's deaths A, S0 = B0 + A0 and lane j's S1_j = B1_j + A1_j, scaled by exp(-M) with M the
//      running maximum of eta over the samples added (online softmax: no risk-set sum is 0 or inf for any finite
//      beta). Closing the group of an event time tau (m deaths) adds, with d0_k = B0 + (1 - f_k) A0 and
//      d1_k = B1 + (1 - f_k) A1 (f_k = k / m for Efron, 0 for Breslow; no subtraction),
//        loglik  sum_D (eta - M) - sum_k log d0_k,
//        U_j     sum_D u_j - B1_j c - A1_j g,    c = sum_k 1 / d0_k, g = sum_k (1 - f_k) / d0_k,
//        I       -(a B1 B1' + b (B1 A1' + A1 B1') + e A1 A1'),   a, b, e = sum_k (1, 1 - f_k, (1 - f_k)^2) / d0_k^2,
//      and stores (tau's group, c, g, M) to the warp's scratch.
//   B  ascending time: Lambda = sum over event times tau <= t_s of c_tau exp(-M_tau), kept relative to the last M,
//      gives W_s = r_s (Lambda_s, or Lambda before t_s + g for a death at t_s) >= 0, and accumulate_tile adds
//      sum_s W_s u_s u_s' = sum_tau sum_k d2_k / d0_k to I (first evaluation: the uncentred I+_jj of the rank rule).
// Every quantity is invariant under adding one constant to every eta and under shifting a column, so the kernel uses
// the centred design. A grid-stride loop over blocks of loci keeps the scratch (n_samples entries per warp slot) fixed.
constexpr int kCMaxIter = 20;                          // coxph.control(iter.max = 20)
constexpr double kCEps = 1e-9;                         // coxph.control(eps = 1e-9)
constexpr double kCTolerInf = 3.1622776601683795e-05;  // coxph.control(toler.inf = sqrt(eps))

template <int P, bool kEfron>
__global__ void __launch_bounds__(kAWarps * 32, 1)
k_assoc_cox(const double *__restrict__ haps, uint64_t n_rows, uint32_t n_all, const uint32_t *__restrict__ idx,
            uint32_t n_samples, uint32_t p, int use_max, const double *__restrict__ design,
            const double *__restrict__ shift, const double *__restrict__ event, const uint32_t *__restrict__ tgroup,
            double4 *scratch, AssocOut out)
{
    __shared__ double s_des[kATile][P + 1];
    __shared__ double s_y[kATile];             // event of the tile's samples
    __shared__ double s_beta[kAWarps][P];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t xcol = p - 1;
    const int n_tiles = (int)((n_samples + kATile - 1) / kATile);
    const uint64_t n_blocks = (n_rows + kAWarps - 1) / kAWarps;
    double4 *scr = scratch + ((uint64_t)blockIdx.x * kAWarps + warp) * n_samples;
    const double ninf = -__longlong_as_double(0x7ff0000000000000ll);
    for (uint64_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const uint64_t row = blk * kAWarps + warp;
        const bool have = row < n_rows;
        const SampleSubset h{reinterpret_cast<const double2 *>(haps + (have ? row : 0) * 2ull * n_all), idx};
        const auto [n, xbar, events] = locus_prepass(h, event, n_samples, use_max, have, lane);

        uint8_t status = INQ_ASSOC_OK;
        bool done = !have;
        if (have && (n == 0 || events == 0.0)) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
        if (lane < P) s_beta[warp][lane] = 0.0;
        const double my_shift = lane == xcol ? xbar : (lane < P ? shift[lane] : 0.0);
        // b / bnew: this lane's coefficient of beta and beta_new; ll: loglik at beta
        double b = 0.0, bnew = 0.0, ll = 0.0;
        uint32_t kmask = 0;
        int iter = 0;
        bool first = true, halving = false;
        for (;;) {
            if (__syncthreads_and(done)) break;
            double G[P];
#pragma unroll
            for (int k = 0; k < P; ++k) G[k] = 0.0;
            double gx = 0.0, U = 0.0, diag = 0.0, lle = 0.0;
            // A: B0, A0 and lane j's B1_j, A1_j scaled by exp(-M); the pending group's sum_D (eta - M), sum_D u_j, m
            double B0 = 0.0, A0 = 0.0, B1 = 0.0, A1 = 0.0, Deta = 0.0, DU = 0.0, M = ninf;
            uint32_t m = 0, cur = 0xffffffffu, ne = 0;
            auto close = [&]() {
                if (m) {
                    double lsum, c, g, a, bb, e;
                    if constexpr (kEfron) {
                        lsum = c = g = a = bb = e = 0.0;
                        for (uint32_t k = 0; k < m; ++k) {
                            const double of = 1.0 - (double)k / (double)m;
                            const double id = 1.0 / fma(of, A0, B0);
                            lsum += log(fma(of, A0, B0));
                            c += id; g = fma(of, id, g);
                            const double id2 = id * id;
                            a += id2; bb = fma(of, id2, bb); e = fma(of * of, id2, e);
                        }
                    } else {
                        const double d0 = B0 + A0, id = 1.0 / d0;
                        lsum = (double)m * log(d0); c = g = (double)m * id; a = bb = e = c * id;
                    }
                    lle += Deta - lsum;
                    U += DU - fma(B1, c, A1 * g);
#pragma unroll
                    for (int k = 0; k < P; ++k) {
                        const double b1k = __shfl_sync(0xffffffffu, B1, k), a1k = __shfl_sync(0xffffffffu, A1, k);
                        const double v = fma(a * B1, b1k, fma(bb, fma(B1, a1k, A1 * b1k), e * A1 * a1k));
                        if (k == (int)xcol) gx -= v;
                        else G[k] -= v;
                    }
                    if (lane == 0) scr[ne] = make_double4((double)cur, c, g, M);
                    ++ne;
                }
                B0 += A0; B1 += A1;
                A0 = A1 = Deta = DU = 0.0;
                m = 0;
            };
            for (int t = n_tiles - 1; t >= 0; --t) {
                const uint32_t s0 = (uint32_t)t * kATile;
                stage_tile<P>(s_des, s_y, design, event, s0, n_samples, tid);
                if (done) continue;
                const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
                const bool valid = xt == xt;
                const double eta = lane_eta<P>(s_beta[warp], s_des[lane], xcol, xt);
                const uint32_t tg = valid ? tgroup[s0 + lane] : 0u;
                // M after this lane's sample is added: the maximum over it, the higher lanes and the later tiles
                double mloc = valid ? eta : ninf;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const double q = __shfl_down_sync(0xffffffffu, mloc, o);
                    if (lane + o < 32) mloc = fmax(mloc, q);
                }
                mloc = fmax(mloc, M);
                const double r = exp(eta - mloc);
                unsigned msk = __ballot_sync(0xffffffffu, valid);
                while (msk) {
                    const int i = 31 - __clz(msk);
                    msk &= ~(1u << i);
                    const uint32_t tgi = __shfl_sync(0xffffffffu, tg, i);
                    if (tgi != cur) { close(); cur = tgi; }
                    const double mi = __shfl_sync(0xffffffffu, mloc, i);
                    if (mi > M) {
                        const double sc = exp(M - mi);
                        B0 *= sc; A0 *= sc; B1 *= sc; A1 *= sc;
                        if (m) Deta -= (double)m * (mi - M);
                        M = mi;
                    }
                    const double ri = __shfl_sync(0xffffffffu, r, i), xi = __shfl_sync(0xffffffffu, xt, i);
                    const double ei = __shfl_sync(0xffffffffu, eta, i);
                    const double uj = lane == xcol ? xi : (lane < P ? s_des[i][lane < P ? lane : 0] : 0.0);
                    if (s_y[i] != 0.0) { A0 += ri; A1 = fma(ri, uj, A1); DU += uj; Deta += ei - M; ++m; }
                    else { B0 += ri; B1 = fma(ri, uj, B1); }
                }
            }
            if (!done) close();
            // B: Lt = Lambda exp(M_c) at the last event time seen, Lp the same before it, gc its g
            double Lt = 0.0, Lp = 0.0, gc = 0.0, Mc = 0.0;
            bool here = false;
            int e = (int)ne - 1;
            cur = 0xffffffffu;
            for (uint32_t s0 = 0; s0 < n_samples; s0 += kATile) {
                stage_tile<P>(s_des, s_y, design, event, s0, n_samples, tid);
                if (done) continue;
                const double xt = lane_x(h, s0 + lane, n_samples, use_max, xbar);
                const bool valid = xt == xt;
                const double eta = lane_eta<P>(s_beta[warp], s_des[lane], xcol, xt);
                const uint32_t tg = valid ? tgroup[s0 + lane] : 0u;
                double lam = 0.0, mref = 0.0;
                unsigned msk = __ballot_sync(0xffffffffu, valid);
                while (msk) {
                    const int i = __ffs(msk) - 1;
                    msk &= msk - 1;
                    const uint32_t tgi = __shfl_sync(0xffffffffu, tg, i);
                    if (tgi != cur) {
                        cur = tgi;
                        here = false;
                        if (e >= 0) {
                            const double4 sc = scr[e];
                            if (sc.x == (double)tgi) {
                                Lp = Lt > 0.0 ? Lt * exp(sc.w - Mc) : 0.0;
                                Lt = Lp + sc.y;
                                gc = sc.z;
                                Mc = sc.w;
                                here = true;
                                --e;
                            }
                        }
                    }
                    if ((int)lane == i) { lam = here && s_y[i] != 0.0 ? Lp + gc : Lt; mref = Mc; }
                }
                // eta <= mref wherever lam > 0: the sample is in the risk set that gave mref
                const double W = lam > 0.0 ? lam * exp(eta - mref) : 0.0;
                double none = 0.0;
                accumulate_tile<P>(G, gx, none, diag, s_des, lane, xcol, valid, xt, W, 0.0, my_shift, first,
                                   [](double &, double, double, double, int) {});
            }
            if (done) continue;
            put_x(G, gx, xcol);
            uint32_t kept = 0;
            double d_x = 0.0, dl[1], r1[1] = {U};
            ldl_solve<P>(G, r1, dl, p, lane, [&](int c, double d) {
                const bool k = first ? c > 0 && d > kAAlias * __shfl_sync(0xffffffffu, diag, c) : ((kmask >> c) & 1u) != 0;
                if (k) { kept |= 1u << c; if (c == (int)xcol) d_x = d; }
                return k;
            });
            const double delta = dl[0];            // this lane's entry of I^-1 U
            if (first) {
                first = false;
                kmask = kept;
                if (n <= (uint32_t)__popc(kept)) { status = INQ_ASSOC_FEW_SAMPLES; done = true; }
                else if (!((kept >> xcol) & 1u)) { status = INQ_ASSOC_SINGULAR; done = true; }
                else { ll = lle; bnew = b + delta; publish_beta<P>(s_beta[warp], lane, bnew); }
                continue;
            }
            ++iter;
            const bool conv = fabs(lle - ll) <= kCEps * fabs(lle) && !halving;
            if (conv || iter == kCMaxIter) {
                const double bx = __shfl_sync(0xffffffffu, bnew, xcol), dx = fabs(__shfl_sync(0xffffffffu, delta, xcol));
                if (!conv) status = INQ_ASSOC_NO_CONVERGENCE;
                else if (dx > kCEps && dx > kCTolerInf * fabs(bx)) status = INQ_ASSOC_SEPARATION;
                if (lane == 0) {
                    const double se = sqrt(1.0 / d_x), zs = bx / se;
                    out.beta[row] = bx; out.se[row] = se; out.stat[row] = zs; out.p[row] = erfc(fabs(zs) * M_SQRT1_2);
                }
                done = true;
                continue;
            }
            if (lle < ll) { halving = true; bnew = 0.5 * (b + bnew); }
            else { halving = false; ll = lle; b = bnew; bnew = b + delta; }
            publish_beta<P>(s_beta[warp], lane, bnew);
        }
        write_tail(out, row, have, lane, n, status, iter);
    }
}

// The Cox launches live in a translation unit of their own (inq_cox_launch.cu): instantiated next to the other assoc
// kernels, k_assoc_cox changed the compiled code of k_assoc_linear_traits.
cudaError_t cox_occupancy(int P, bool efron, int *per_sm);
void cox_launch(int P, bool efron, unsigned grid, cudaStream_t s, const double *haps, uint64_t n_rows, uint32_t n_all,
                const uint32_t *idx, uint32_t n_samples, uint32_t p, int use_max, const double *design, const double *shift,
                const double *event, const uint32_t *tgroup, double4 *scratch, AssocOut out);

}  // namespace inqa
