"""numpy/scipy restatement of `inquistr-b200 assoc` (DESIGN.md 5e): per-locus linear (OLS, Student t) and logistic
(IRLS as R's glm.fit without step-halving, Wald z) regression of a trait on STR length, design [1, covariates..., x].

Independent of the kernel's arithmetic: rank decisions come from a Householder QR of the weighted design,
the fits from np.linalg.lstsq on the uncentred design, the standard error from a Householder QR, the p-values from
scipy.stats. Test infrastructure only."""
from __future__ import annotations

import numpy as np
from scipy import stats

OK, FEW_SAMPLES, SINGULAR, NO_CONVERGENCE, SEPARATION = 0, 1, 2, 3, 4
STATUS_NAMES = ["ok", "few_samples", "singular", "no_convergence", "separation"]
ALIAS = 1e-10
MAX_ITER = 25
EPSILON = 1e-8
DBL_EPS = np.finfo(np.float64).eps


def predictor(h1, h2, mode="sum"):
    h1 = np.asarray(h1, np.float64)
    h2 = np.asarray(h2, np.float64)
    if mode == "sum":
        return h1 + h2
    return np.fmax(h1, h2)                          # NaN only when both are NaN


def linkinv(eta):
    return linkinv2(eta)[0]


def linkinv2(eta):
    """(mu, 1 - mu), the second as 1 / (1 + t) rather than by subtraction (no cancellation near mu = 1)."""
    t = np.where(eta < -30, DBL_EPS, np.where(eta > 30, 1 / DBL_EPS, np.exp(np.clip(eta, -30, 30))))
    return t / (1 + t), 1 / (1 + t)


def mu_eta(eta):
    e = np.exp(np.clip(eta, -30, 30))
    return np.where(np.abs(eta) > 30, DBL_EPS, e / ((1 + e) * (1 + e)))


def kept_columns(X, w):
    """The rank rule: column j is aliased when the weighted residual sum of squares of column j after the kept
    earlier columns (its elimination pivot) is <= 1e-10 * sum(w * X_j^2). The residuals are R_jj^2 of a Householder
    QR of sqrt(w) X; once a column is dropped, each later column gets a QR of the kept columns and itself."""
    A = np.sqrt(w)[:, None] * X
    R = np.linalg.qr(A, mode="r")
    keep = []
    for j in range(X.shape[1]):
        if len(keep) == j:
            d = R[j, j] ** 2 if j < R.shape[0] else 0.0
        else:
            Rj = np.linalg.qr(A[:, keep + [j]], mode="r")
            d = Rj[-1, -1] ** 2 if len(keep) < Rj.shape[0] else 0.0
        if d > ALIAS * float(A[:, j] @ A[:, j]):
            keep.append(j)
    return keep


def _wls(X, w, z):
    keep = kept_columns(X, w)
    xcol = X.shape[1] - 1
    sw = np.sqrt(w)
    A = sw[:, None] * X[:, keep]
    coef = np.linalg.lstsq(A, sw * z, rcond=None)[0]
    beta = np.zeros(X.shape[1])
    beta[keep] = coef
    ginv_xx = np.nan
    if keep and keep[-1] == xcol:
        R = np.linalg.qr(A, mode="r")
        ginv_xx = 1.0 / R[-1, -1] ** 2                # x last: (A'A)^-1_xx = 1 / R_xx^2
    return keep, beta, ginv_xx


def fit_locus(x, y, cov=None, model="linear"):
    """-> dict(beta, se, stat, p, n, status, n_iter, coef) for one locus; x has NaN for samples without a call;
    coef: every coefficient of [1, covariates..., x] (0 for a dropped column), None where no fit is reported."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    ns = len(y)
    cov = np.zeros((ns, 0)) if cov is None else np.asarray(cov, np.float64).reshape(ns, -1)
    use = ~np.isnan(x)
    n = int(use.sum())
    res = dict(beta=np.nan, se=np.nan, stat=np.nan, p=np.nan, n=n, status=FEW_SAMPLES, n_iter=0, coef=None)
    if n == 0:
        return res
    X = np.column_stack([np.ones(n), cov[use], x[use]])
    yy = y[use]
    if model == "linear":
        keep, beta, g = _wls(X, np.ones(n), yy)
        if n <= len(keep):
            return res
        if X.shape[1] - 1 not in keep:
            res["status"] = SINGULAR
            return res
        r = yy - X @ beta
        df = n - len(keep)
        se = np.sqrt(float(r @ r) / df * g)
        t = beta[-1] / se
        res.update(beta=beta[-1], se=se, stat=t, p=2 * stats.t.sf(abs(t), df), status=OK, coef=beta)
        return res
    if yy.min() == yy.max():
        return res                                    # one class
    mu = (yy + 0.5) / 2
    eta = np.log(mu / (1 - mu))
    mu, omu = linkinv2(eta)

    def deviance(mu, omu):
        return float(np.sum(np.where(yy != 0, -2 * np.log(mu), -2 * np.log(omu))))

    dev_old = deviance(mu, omu)
    g = np.nan
    for it in range(1, MAX_ITER + 1):
        me = mu_eta(eta)
        w = me * me / (mu * omu)
        z = eta + np.where(yy != 0, omu, -mu) / me
        keep, beta, g = _wls(X, w, z)
        if it == 1 and n <= len(keep):
            return res
        if X.shape[1] - 1 not in keep:
            res.update(status=SINGULAR, n_iter=it - 1)
            return res
        eta = X @ beta
        mu, omu = linkinv2(eta)
        dev = deviance(mu, omu)
        conv = abs(dev - dev_old) / (abs(dev) + 0.1) < EPSILON
        dev_old = dev
        if conv:
            break
    status = OK
    if not conv:
        status = NO_CONVERGENCE
    elif np.any(mu < 10 * DBL_EPS) or np.any(omu < 10 * DBL_EPS):
        status = SEPARATION
    se = np.sqrt(g)
    zs = beta[-1] / se
    res.update(beta=beta[-1], se=se, stat=zs, p=2 * stats.norm.sf(abs(zs)), status=status, n_iter=it, coef=beta)
    return res


def assoc_matrix(haps, y, cov=None, model="linear", predictor_mode="sum"):
    """Every row of haps (rows x 2 * samples: H1, H2 per sample) -> dict of per-row arrays."""
    haps = np.asarray(haps, np.float64)
    rows = haps.shape[0]
    out = {k: np.full(rows, np.nan) for k in ("beta", "se", "stat", "p")}
    out["n"] = np.zeros(rows, np.int64)
    out["status"] = np.zeros(rows, np.int64)
    out["n_iter"] = np.zeros(rows, np.int64)
    for i in range(rows):
        x = predictor(haps[i, 0::2], haps[i, 1::2], predictor_mode)
        r = fit_locus(x, y, cov, model)
        for k in ("beta", "se", "stat", "p", "n", "status", "n_iter"):
            out[k][i] = r[k]
    return out
