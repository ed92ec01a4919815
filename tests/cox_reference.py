"""numpy/scipy restatement of `inquistr-b200 assoc --model cox` (DESIGN.md 5e, Cox), independent of the kernel's
arithmetic: Cox proportional hazards with Efron or Breslow ties, Newton iteration with coxph.fit's control flow
(coxfit6). Written from the definition: one explicit risk set per distinct event time, the risk-set sums through
scipy.special.logsumexp, np.linalg solves, the rank rule from Schur complements. Design u = [covariates..., x] (no
intercept), uncentred. The predictor, the statuses and the aliasing tolerance are oracle/assoc.py's. Test
infrastructure only."""
from __future__ import annotations

import numpy as np
from scipy import stats
from scipy.special import logsumexp

from oracle.assoc import ALIAS, FEW_SAMPLES, NO_CONVERGENCE, OK, SEPARATION, SINGULAR, predictor

COX_EPS = 1e-9                  # coxph.control(eps = 1e-9)
COX_MAX_ITER = 20               # coxph.control(iter.max = 20)
COX_TOLER_INF = COX_EPS ** 0.5  # coxph.control(toler.inf = sqrt(eps))


def cox_evaluate(U, time, event, beta, ties="efron"):
    """-> (loglik, score, information, uncentred diagonal) of the partial likelihood at beta.
    The diagonal is sum over event times and Efron steps k of (d2_k)_jj / d0_k, the I+_jj of the rank rule."""
    q = U.shape[1]
    eta = U @ beta
    ll, score, info, diag = 0.0, np.zeros(q), np.zeros((q, q)), np.zeros(q)
    for tau in np.unique(time[event != 0]):
        R = time >= tau
        dead = (time == tau) & (event != 0)
        m = int(dead.sum())
        uR, eR, dR = U[R], eta[R], dead[R]
        f = np.arange(m) / m if ties == "efron" else np.zeros(m)
        # weights of the m Efron steps over the risk set: r_i (1 - f_k [i died at tau])
        b = 1.0 - f[:, None] * dR[None, :]                                    # m x |R|
        logd0 = logsumexp(np.broadcast_to(eR, b.shape), axis=1, b=b)          # log d0_k
        p = b * np.exp(eR[None, :] - logd0[:, None])                          # p_ki, rows sum to 1
        mu = p @ uR                                                           # d1_k / d0_k
        ll += float(eta[dead].sum() - logd0.sum())
        score += U[dead].sum(axis=0) - mu.sum(axis=0)
        # sum_k cov_k, centred at mu_0: sum_i q_i (u_i - c)(u_i - c)' - sum_k (mu_k - c)(mu_k - c)'
        c = mu[0]
        qi = p.sum(axis=0)
        dc = uR - c
        info += (dc * qi[:, None]).T @ dc - (mu - c).T @ (mu - c)
        diag += qi @ (uR * uR)
    return ll, score, info, diag


def cox_kept_columns(info, diag):
    """The rank rule on I at beta = 0: column j is aliased when its Schur complement after the kept earlier columns,
    I_jj - I_jK I_KK^-1 I_Kj, is <= 1e-10 * I+_jj."""
    keep = []
    for j in range(info.shape[0]):
        d = info[j, j]
        if keep:
            d -= float(info[j, keep] @ np.linalg.solve(info[np.ix_(keep, keep)], info[keep, j]))
        if d > ALIAS * diag[j]:
            keep.append(j)
    return keep


def fit_locus_cox(x, time, event, cov=None, ties="efron"):
    """-> dict(beta, se, stat, p, n, status, n_iter, coef) for one locus: Cox regression of (time, event) on
    [covariates..., x]; x has NaN for samples without a call. stat is the Wald z, coef every coefficient (0 for a
    dropped column), None where no fit is reported."""
    x = np.asarray(x, np.float64)
    time = np.asarray(time, np.float64)
    event = np.asarray(event, np.float64)
    ns = len(time)
    cov = np.zeros((ns, 0)) if cov is None else np.asarray(cov, np.float64).reshape(ns, -1)
    use = ~np.isnan(x)
    n = int(use.sum())
    res = dict(beta=np.nan, se=np.nan, stat=np.nan, p=np.nan, n=n, status=FEW_SAMPLES, n_iter=0, coef=None)
    t, d = time[use], event[use]
    if n == 0 or not np.any(d != 0):
        return res
    U = np.column_stack([cov[use], x[use]])
    q = U.shape[1]
    beta = np.zeros(q)
    ll, score, info, diag = cox_evaluate(U, t, d, beta, ties)
    keep = cox_kept_columns(info, diag)
    if n <= len(keep):
        return res
    if q - 1 not in keep:
        res["status"] = SINGULAR
        return res

    def step(score, info):
        delta = np.zeros(q)
        delta[keep] = np.linalg.solve(info[np.ix_(keep, keep)], score[keep])
        return delta

    beta_new = beta + step(score, info)
    halving = False
    for it in range(1, COX_MAX_ITER + 1):
        ll_new, score, info, _ = cox_evaluate(U, t, d, beta_new, ties)
        if abs(ll_new - ll) <= COX_EPS * abs(ll_new) and not halving:
            status = OK
            break
        if it == COX_MAX_ITER:
            status = NO_CONVERGENCE
            break
        if ll_new < ll:
            halving = True
            beta_new = (beta + beta_new) / 2
        else:
            halving = False
            ll, beta = ll_new, beta_new
            beta_new = beta + step(score, info)
    ik = np.linalg.inv(info[np.ix_(keep, keep)])
    se = float(np.sqrt(ik[-1, -1]))
    if status == OK:
        inf_x = abs(float(ik[-1] @ score[keep]))
        if inf_x > COX_EPS and inf_x > COX_TOLER_INF * abs(beta_new[-1]):
            status = SEPARATION
    z = beta_new[-1] / se
    res.update(beta=float(beta_new[-1]), se=se, stat=z, p=float(2 * stats.norm.sf(abs(z))), status=status, n_iter=it,
               coef=beta_new)
    return res


def assoc_cox_matrix(haps, time, event, cov=None, ties="efron", predictor_mode="sum"):
    """Every row of haps (rows x 2 * samples: H1, H2 per sample) -> dict of per-row arrays, as assoc_matrix."""
    haps = np.asarray(haps, np.float64)
    rows = haps.shape[0]
    out = {k: np.full(rows, np.nan) for k in ("beta", "se", "stat", "p")}
    for k in ("n", "status", "n_iter"):
        out[k] = np.zeros(rows, np.int64)
    for i in range(rows):
        x = predictor(haps[i, 0::2], haps[i, 1::2], predictor_mode)
        r = fit_locus_cox(x, time, event, cov, ties)
        for k in out:
            out[k][i] = r[k]
    return out
