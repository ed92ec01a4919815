/* inqcohort.h -- C ABI of the cohort `outlier` rows (SURVEY.md 8f rank 3), part of libinqcall.so.
 *
 * Replaces the per-line body of the reference's `outlier` loop (src/outlier.rs:41-71, wdecoster/inquiSTR
 * v0.13.0) for a whole combined matrix at once: rows = loci, columns = the haplotype columns
 * `<sample>_H1, <sample>_H2, ...` of the `combine` TSV (combine.rs:27-59), values = f32 as parsed by
 * outlier.rs:76-80. There is no CPU implementation behind these entry points.
 *
 *   get_repeat_lengths   outlier.rs:75-97   NaN -> 0, row dropped when max < minsize
 *   z_score_outliers     outlier.rs:18-31,99-113  f32 sequential mean / population sd, (v - mean) / sd >= cutoff
 *   dbscan_outliers      outlier.rs:115-145 + dbscan 0.3.1   eps = max(2 * mode, 10), min_points = ilog2(columns),
 *                        outliers = Noise
 * What the caller keeps: the sample names (suffix stripping outlier.rs:112,130), --subset filtering
 * (outlier.rs:59-67) and the TSV text.
 *
 * inq_assoc: per-locus association of STR length with a trait (`inquistr-b200 assoc`, DESIGN.md 5e); the model is
 * this project's own (the reference has it only as an external R script): OLS with a Student t test, or logistic
 * IRLS as R's glm.fit without step-halving with a Wald z test, or Firth-penalized logistic regression with a penalized
 * likelihood-ratio test; design [1, covariates..., x], x last. inq_assoc_cox fits Cox proportional hazards of a
 * censored time (age at onset) instead.
 */
#ifndef INQCOHORT_H
#define INQCOHORT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INQ_OUTLIER_ZSCORE 0       /* outlier.rs Method::Zscore */
#define INQ_OUTLIER_DBSCAN 1       /* outlier.rs Method::Dbscan */

#define INQ_ERR_NO_MODE (-15)      /* dbscan: a kept row without a positive value (the reference panics, outlier.rs:144) */
#define INQ_ERR_HITS_CAP (-16)     /* more outliers than `cap`: *n_hits holds the number needed */

/* Flags the outliers of every row of `values` (host memory, row-major n_rows x n_cols, NaN allowed).
 *   row_kept : n_rows bytes, 1 = the row passed the minsize test (nullable)
 *   hits     : up to `cap` entries (row << 32 | column), sorted ascending = the reference's print order
 *   n_hits   : number of outliers found (also set on INQ_ERR_HITS_CAP)
 * Returns 0 or a negative INQ_ERR_* code (inqcall.h); inq_cohort_last_error() describes the failure. */
int inq_outlier(int device, int method, uint64_t n_rows, uint32_t n_cols, const float *values,
                uint32_t minsize, float zscore_cutoff, uint8_t *row_kept,
                uint64_t *n_hits, uint64_t *hits, uint64_t cap, float *ms_kernel /* nullable */);

#define INQ_ASSOC_LINEAR 0         /* OLS, t test with n - rank degrees of freedom */
#define INQ_ASSOC_LOGISTIC 1       /* binomial / logit IRLS, Wald z test, dispersion 1 */
#define INQ_ASSOC_FIRTH 2          /* Firth-penalized logit (Jeffreys prior), penalized likelihood-ratio chi^2 test */
#define INQ_ASSOC_SUM 0            /* predictor H1 + H2, missing if either is NaN */
#define INQ_ASSOC_MAX 1            /* predictor max of the non-NaN alleles, missing if both are NaN */

#define INQ_ASSOC_OK 0
#define INQ_ASSOC_FEW_SAMPLES 1    /* n <= rank, or (logistic) only one class among the samples used */
#define INQ_ASSOC_SINGULAR 2       /* x aliased by the intercept and covariates */
#define INQ_ASSOC_NO_CONVERGENCE 3 /* logistic: 25 iterations without meeting the deviance criterion;
                                      firth: the full or the null fit took 100 steps without converging */
#define INQ_ASSOC_SEPARATION 4     /* logistic: a fitted probability below 10 eps or above 1 - 10 eps (never for firth) */

#define INQ_ASSOC_MAX_COV 30       /* design columns: intercept + covariates + x <= 32 */

/* Tests every row of `haps` (host memory, row-major n_rows x 2 * n_samples f64: H1, H2 of each sample, NaN = no
 * call) for association with the trait `y[n_samples]` (logistic and firth: every value 0 or 1), adjusted for the
 * covariates `cov` (row-major n_samples x n_cov, no missing values). Per row: beta, se, stat (t or z), two-sided p
 * (NaN when the status is FEW_SAMPLES or SINGULAR), n_used (samples with a predictor) and status (INQ_ASSOC_*);
 * n_iter (nullable) is the number of weighted solves of a logistic fit (0 for linear).
 * INQ_ASSOC_FIRTH: beta and se = sqrt((I^-1)_xx) of the penalized full fit, stat the penalized likelihood-ratio
 * chi^2 (full against x = 0, both fits penalized by the full model's log det I), p from chi^2 with 1 df, and n_iter
 * the full fit's number of steps.
 * Returns 0 or a negative INQ_ERR_* code (inqcall.h); inq_cohort_last_error() describes the failure. */
int inq_assoc(int device, int model, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
              const double *y, uint32_t n_cov, const double *cov, double *beta, double *se, double *stat, double *p,
              uint32_t *n_used, uint8_t *status, uint8_t *n_iter /* nullable */, float *ms_kernel /* nullable */);

/* Several traits at once: every trait t (column t of y, row-major n_samples x n_traits, NaN = the sample is not used
 * for t; logistic and firth: every other value 0 or 1; +-inf is rejected) gives, in column t of the row-major
 * n_rows x n_traits outputs, exactly what inq_assoc gives for t alone over the samples where y is not NaN (bit for bit).
 * All traits share the model, the predictor and the covariates (finite, as in inq_assoc). The haplotype matrix goes
 * to the device once; traits with the same samples share one preparation, and the linear ones one Gram matrix per
 * locus. ms_kernel is the summed kernel time of all sample sets.
 * INQ_ERR_ARG for n_traits == 0 and for a trait without a value (the message names the trait index);
 * INQ_ERR_TOO_LARGE when n_rows x n_traits does not fit in memory sizes, or one sample set's loci x traits exceed the
 * launch shape (2^31 - 1 blocks of 4 loci for logistic and firth; of 4 loci and up to 4 to 16 linear traits (by the design width)). */
int inq_assoc_traits(int device, int model, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
                     uint32_t n_traits, const double *y, uint32_t n_cov, const double *cov, double *beta, double *se,
                     double *stat, double *p, uint32_t *n_used, uint8_t *status, uint8_t *n_iter /* nullable */,
                     float *ms_kernel /* nullable */);

#define INQ_COX_EFRON 0            /* Efron's approximation for tied event times (coxph's default) */
#define INQ_COX_BRESLOW 1          /* Breslow's approximation */

/* Cox proportional-hazards regression of a censored time on STR length (`assoc --model cox`, DESIGN.md 5e, Cox), as
 * R's coxph(Surv(time, event) ~ covariates + x) with ties = "efron" or "breslow" and coxph.control's defaults:
 * partial likelihood over u = [covariates..., x] (no intercept), Newton iteration with step-halving, at most 20
 * iterations, converged when |loglik - loglik_old| <= 1e-9 |loglik|. time[n_samples]: any finite number;
 * event[n_samples]: 1 = event at that time, 0 = censored at it (still at risk there). Per row: beta and
 * se = sqrt((I^-1)_xx) of the fit, stat the Wald z, p = erfc(|z| / sqrt 2), n_used and status as inq_assoc, and
 * n_iter (nullable) the Newton iterations. Statuses: FEW_SAMPLES (no event among the samples used, or n <= rank),
 * SINGULAR, NO_CONVERGENCE (20 iterations), SEPARATION (a converged fit whose last Newton step for x, |(I^-1 U)_x|,
 * exceeds 1e-9 and sqrt(1e-9) |beta|: the coefficient may be infinite, coxph's toler.inf rule).
 * INQ_ERR_ARG names the sample for a non-finite time or covariate and an event that is not 0 or 1;
 * INQ_ERR_TOO_LARGE when the rows exceed the launch shape (2^31 - 1 blocks of 4 loci). */
int inq_assoc_cox(int device, int ties, int predictor, uint64_t n_rows, uint32_t n_samples, const double *haps,
                  const double *time, const uint8_t *event, uint32_t n_cov, const double *cov, double *beta, double *se,
                  double *stat, double *p, uint32_t *n_used, uint8_t *status, uint8_t *n_iter /* nullable */,
                  float *ms_kernel /* nullable */);

const char *inq_cohort_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
