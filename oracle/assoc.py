"""numpy/scipy restatement of `inquistr-b200 assoc` (DESIGN.md 5e): per-locus linear (OLS, Student t), logistic
(IRLS as R's glm.fit without step-halving, Wald z) and Firth-penalized logistic (penalized likelihood-ratio test,
`--firth`) regression of a trait on STR length, design [1, covariates..., x].

Independent of the kernel's arithmetic: rank decisions come from a Householder QR of the weighted design,
the fits from np.linalg.lstsq on the uncentred design, the standard error from a Householder QR, the p-values from
scipy.stats. Firth fits the uncentred design too: the rank set comes from `kept_columns` with equal weights, h_i
from the row sums of Q^2 of a QR of W^1/2 X_K, log det I from `slogdet` of that QR's R, the step from
np.linalg.lstsq, p from scipy.stats.chi2. Test infrastructure only."""
from __future__ import annotations

import numpy as np
from scipy import stats

OK, FEW_SAMPLES, SINGULAR, NO_CONVERGENCE, SEPARATION = 0, 1, 2, 3, 4
STATUS_NAMES = ["ok", "few_samples", "singular", "no_convergence", "separation"]
ALIAS = 1e-10
MAX_ITER = 25
EPSILON = 1e-8
DBL_EPS = np.finfo(np.float64).eps
MAX_STEPS = 100                 # Firth: steps per fit
MAX_HALVINGS = 5                # Firth: halvings per step
LAMBDA2 = 1e-10                 # Firth: converged when delta_F . U*_F falls below this
RISE = 1e-12                    # Firth: a step is halved when D* rises by more than RISE * (|D*_prev| + 1)


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


def _evaluate(X, y, beta):
    """Firth, at beta: (penalized deviance D*, mu, 1 - mu, w, Q of W^1/2 X_K, R of it)."""
    mu, omu = linkinv2(X @ beta)
    w = mu * omu
    Q, R = np.linalg.qr(np.sqrt(w)[:, None] * X, mode="reduced")
    logdet = 2 * np.linalg.slogdet(R)[1]               # log det (X' W X) = log det R'R
    dev = -2 * float(np.sum(np.where(y != 0, np.log(mu), np.log(omu))))
    return dev - logdet, mu, omu, w, Q, R


def _fit(XK, y, free):
    """One Firth fit over the free columns `free` (indices into XK); the others stay 0.
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


def _firth(X, yy, res):
    """The full and the null Firth fit of one locus with at least one case and one control; fills res."""
    n = X.shape[0]
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


def fit_locus(x, y, cov=None, model="linear"):
    """-> dict(beta, se, stat, p, n, status, n_iter, coef) for one locus; x has NaN for samples without a call;
    model: "linear", "logistic" or "firth", as cohort.assoc; coef: every coefficient of [1, covariates..., x]
    (0 for a dropped column), None where no fit is reported. firth: stat is the penalized likelihood-ratio chi^2
    (1 df), n_iter the full fit's steps, and the dict also has the null fit's n_iter_null and coef_null."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    ns = len(y)
    cov = np.zeros((ns, 0)) if cov is None else np.asarray(cov, np.float64).reshape(ns, -1)
    use = ~np.isnan(x)
    n = int(use.sum())
    res = dict(beta=np.nan, se=np.nan, stat=np.nan, p=np.nan, n=n, status=FEW_SAMPLES, n_iter=0, coef=None)
    if model == "firth":
        res.update(n_iter_null=0, coef_null=None)
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
    if model == "firth":
        return _firth(X, yy, res)
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
    """Every row of haps (rows x 2 * samples: H1, H2 per sample) -> dict of per-row arrays (firth: with n_iter_null)."""
    haps = np.asarray(haps, np.float64)
    rows = haps.shape[0]
    out = {k: np.full(rows, np.nan) for k in ("beta", "se", "stat", "p")}
    counts = ("n", "status", "n_iter") + (("n_iter_null",) if model == "firth" else ())
    for k in counts:
        out[k] = np.zeros(rows, np.int64)
    for i in range(rows):
        x = predictor(haps[i, 0::2], haps[i, 1::2], predictor_mode)
        r = fit_locus(x, y, cov, model)
        for k in ("beta", "se", "stat", "p") + counts:
            out[k][i] = r[k]
    return out
