"""numpy/scipy restatement of `inquistr-b200 assoc --firth` (DESIGN.md 5e, Firth): Firth-penalized logistic
regression of a trait on STR length, design [1, covariates..., x], with a penalized likelihood-ratio test.

Independent of the kernel's arithmetic: it fits the uncentred design; the rank set comes from `kept_columns` of
oracle/assoc.py with equal weights; h_i from the row sums of Q^2 of a QR of W^1/2 X_K; log det I from `slogdet` of
that QR's R; the step from np.linalg.lstsq; p from scipy.stats.chi2. The existing `oracle/assoc.py` is reused for the
link, the predictor and the rank rule only. Test infrastructure only."""
from __future__ import annotations

import numpy as np
from scipy import stats

from oracle.assoc import FEW_SAMPLES, NO_CONVERGENCE, OK, SINGULAR, kept_columns, linkinv2, predictor

MAX_STEPS = 100                 # steps per fit
MAX_HALVINGS = 5                # halvings per step
LAMBDA2 = 1e-10                 # converged when delta_F . U*_F falls below this
RISE = 1e-12                    # a step is halved when D* rises by more than RISE * (|D*_prev| + 1)


def _evaluate(X, y, beta):
    """At beta: (penalized deviance D*, mu, 1 - mu, w, Q of W^1/2 X_K, R of it)."""
    mu, omu = linkinv2(X @ beta)
    w = mu * omu
    Q, R = np.linalg.qr(np.sqrt(w)[:, None] * X, mode="reduced")
    logdet = 2 * np.linalg.slogdet(R)[1]               # log det (X' W X) = log det R'R
    dev = -2 * float(np.sum(np.where(y != 0, np.log(mu), np.log(omu))))
    return dev - logdet, mu, omu, w, Q, R


def _fit(XK, y, free):
    """One fit over the free columns `free` (indices into XK); the others stay 0.
    -> (beta, D*, R of the last evaluation, steps, converged)."""
    beta = np.zeros(XK.shape[1])
    beta_prev, d_prev = beta, 0.0
    t = halvings = 0
    while True:
        d, mu, omu, w, Q, R = _evaluate(XK, y, beta)
        if t > 0 and d > d_prev + RISE * (abs(d_prev) + 1) and halvings < MAX_HALVINGS:
            beta = (beta + beta_prev) / 2
            halvings += 1
            continue
        h = np.sum(Q * Q, axis=1)                                      # w_i x_i' I^-1 x_i
        r = np.where(y != 0, omu, -mu) + h * (0.5 - mu)                # y - mu + h (1/2 - mu)
        s = np.sqrt(w * (1 + h))
        # delta_F = H_FF^-1 U*_F with H = X' diag(w (1 + h)) X and U* = X' r: least squares of (s X_F) delta = r / s
        delta_f = np.linalg.lstsq(s[:, None] * XK[:, free], r / s, rcond=None)[0]
        lam2 = float(delta_f @ (XK[:, free].T @ r))
        if lam2 < LAMBDA2:
            return beta, d, R, t, True
        if t == MAX_STEPS:
            return beta, d, R, t, False
        beta_prev, d_prev = beta, d
        beta = beta.copy()
        beta[free] += delta_f
        t += 1
        halvings = 0


def fit_locus(x, y, cov=None):
    """-> dict(beta, se, stat, p, n, status, n_iter, n_iter_null, coef, coef_null) for one locus; x has NaN for samples
    without a call. stat is the penalized likelihood-ratio chi^2 (1 df); n_iter / n_iter_null the full / null fit's
    steps; coef / coef_null every coefficient of [1, covariates..., x] of the full and the null fit (0 for a dropped
    column), None without a fit."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    ns = len(y)
    cov = np.zeros((ns, 0)) if cov is None else np.asarray(cov, np.float64).reshape(ns, -1)
    use = ~np.isnan(x)
    n = int(use.sum())
    res = dict(beta=np.nan, se=np.nan, stat=np.nan, p=np.nan, n=n, status=FEW_SAMPLES, n_iter=0, n_iter_null=0,
               coef=None, coef_null=None)
    if n == 0:
        return res
    yy = y[use]
    if yy.min() == yy.max():
        return res                                    # one class
    X = np.column_stack([np.ones(n), cov[use], x[use]])
    xcol = X.shape[1] - 1
    keep = kept_columns(X, np.ones(n))                # decided once, at beta = 0 (equal weights)
    if n <= len(keep):
        return res
    if xcol not in keep:
        res["status"] = SINGULAR
        return res
    XK = X[:, keep]
    b1, d1, R1, t1, c1 = _fit(XK, yy, list(range(len(keep))))
    b0, d0, _, t0, c0 = _fit(XK, yy, list(range(len(keep) - 1)))
    stat = max(0.0, d0 - d1)
    coef, coef_null = np.zeros(X.shape[1]), np.zeros(X.shape[1])
    coef[keep], coef_null[keep] = b1, b0
    res.update(beta=b1[-1], se=1.0 / abs(R1[-1, -1]), stat=stat, p=float(stats.chi2.sf(stat, 1)),
               status=OK if c1 and c0 else NO_CONVERGENCE, n_iter=t1, n_iter_null=t0, coef=coef, coef_null=coef_null)
    return res


def assoc_matrix(haps, y, cov=None, predictor_mode="sum"):
    """Every row of haps (rows x 2 * samples: H1, H2 per sample) -> dict of per-row arrays."""
    haps = np.asarray(haps, np.float64)
    rows = haps.shape[0]
    out = {k: np.full(rows, np.nan) for k in ("beta", "se", "stat", "p")}
    for k in ("n", "status", "n_iter", "n_iter_null"):
        out[k] = np.zeros(rows, np.int64)
    for i in range(rows):
        r = fit_locus(predictor(haps[i, 0::2], haps[i, 1::2], predictor_mode), y, cov)
        for k in ("beta", "se", "stat", "p", "n", "status", "n_iter", "n_iter_null"):
            out[k][i] = r[k]
    return out
