"""Float64 restatement of model comparison: pointwise log-likelihood, WAIC and PSIS-LOO.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

* ``pointwise_loglik``: ``ll[s, m] = log Pois(yh; lh) + log Pois(ya; la) + log tau`` from ``predict.expected_goals``,
  ``predict.correlation_term`` (tau clamped at 0) and ``predict._pois_lp``: the predict path, no weights, no clip of the
  rates.
* ``psislw`` / ``gpdfit``: ArviZ's ``_psislw`` / ``_gpdfit`` (Vehtari et al., "Pareto Smoothed Importance Sampling",
  JMLR 2024; Zhang & Stephens 2009), step for step.  One addition: with S = 1 there is no (Mt+1)-th largest value and
  the cut is log(DBL_MIN) (the tail then has one value, so k-hat = inf and nothing is smoothed).
* ``loo`` / ``waic``: per-match values and totals from an ``[S, M]`` matrix.
"""
from __future__ import annotations

import numpy as np
from scipy.special import logsumexp

from . import predict as op

LOG_TINY = float(np.log(np.finfo(float).tiny))
EPS = float(np.finfo(float).eps)


def pointwise_loglik(model, samples, home, away, home_goals, away_goals, **fx):
    """``[S, M]`` float64 log-likelihood of the observed scores under each posterior draw."""
    lh, la = op.expected_goals(model, samples, home, away, **fx)
    cc = np.asarray(samples["corr_coef"], dtype=np.float64)
    hg = np.asarray(home_goals).astype(np.float64)
    ag = np.asarray(away_goals).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return op._pois_lp(hg, lh) + op._pois_lp(ag, la) + op.correlation_term(hg, ag, lh, la, cc)


def tail_length(S, r_eff=1.0):
    return int(np.ceil(min(0.2 * S, 3 * np.sqrt(S / r_eff))))


def gpdfit(z):
    """Generalised Pareto fit to the ascending values ``z``: returns (k-hat with the weak prior, sigma)."""
    n = len(z)
    m = 30 + int(n ** 0.5)
    b = 1 - np.sqrt(m / (np.arange(1, m + 1, dtype=float) - 0.5))
    b /= 3 * z[int(n / 4 + 0.5) - 1]
    b += 1 / z[-1]
    k = np.log1p(-b[:, None] * z).mean(axis=1)
    L = n * (np.log(-(b / k)) - k - 1)
    w = 1 / np.exp(L - L[:, None]).sum(axis=1)
    keep = w >= 10 * EPS
    w, b = w[keep], b[keep]
    w = w / w.sum()
    bh = np.sum(b * w)
    k = np.log1p(-bh * z).mean()
    sigma = -k / bh
    return (n * k + 10 * 0.5) / (n + 10), sigma


def gpinv(p, k, sigma):
    if not sigma > 0:
        return np.full_like(p, np.nan)
    x = -np.log1p(-p) if abs(k) < EPS else np.expm1(-k * np.log1p(-p)) / k
    return x * sigma


def psislw(log_ratios, r_eff=1.0):
    """Smoothed, normalised log-weights and k-hat of one vector of log importance ratios."""
    x = np.array(log_ratios, dtype=np.float64)
    S = len(x)
    x -= x.max()
    Mt = tail_length(S, r_eff)
    xs = np.sort(x)
    x_cut = max(xs[-Mt - 1] if Mt + 1 <= S else -np.inf, LOG_TINY)
    tail = np.flatnonzero(x > x_cut)
    n = len(tail)
    if n <= 4:
        k = np.inf
    else:
        si = np.argsort(x[tail], kind="stable")
        z = np.exp(x[tail]) - np.exp(x_cut)
        with np.errstate(divide="ignore", invalid="ignore"):
            k, sigma = gpdfit(z[si])
        if np.isfinite(k):
            x[tail[si]] = np.log(gpinv(np.arange(0.5, n) / n, k, sigma) + np.exp(x_cut))
            x[x > 0] = 0
    x -= logsumexp(x)
    return x, k


def loo_pointwise(ll, r_eff=1.0):
    """``ll [S, M]`` -> (elpd_loo_m [M], k-hat [M]); a column with a non-finite entry gives (NaN, inf)."""
    ll = np.asarray(ll, dtype=np.float64)
    M = ll.shape[1]
    elpd, khat = np.empty(M), np.empty(M)
    for m in range(M):
        col = ll[:, m]
        if not np.isfinite(col).all():
            elpd[m], khat[m] = np.nan, np.inf
            continue
        lw, khat[m] = psislw(-col, r_eff)
        elpd[m] = logsumexp(lw + col)
    return elpd, khat


def lppd_pointwise(ll):
    ll = np.asarray(ll, dtype=np.float64)
    return logsumexp(ll, axis=0) - np.log(ll.shape[0])


def waic(ll):
    """Totals of WAIC with the variance over draws at divisor S."""
    lppd = lppd_pointwise(ll)
    p = np.asarray(ll, dtype=np.float64).var(axis=0)
    e = lppd - p
    return {"elpd_waic": e.sum(), "p_waic": p.sum(), "lppd": lppd.sum(), "se": np.sqrt(len(e) * e.var()),
            "pointwise": e}


def loo(ll, r_eff=1.0):
    """Totals of PSIS-LOO: elpd_loo, se = sqrt(M var0(elpd_m)), p_loo = lppd - elpd_loo, and the k-hat counts."""
    ll = np.asarray(ll, dtype=np.float64)
    S = ll.shape[0]
    e, k = loo_pointwise(ll, r_eff)
    lppd = lppd_pointwise(ll)
    with np.errstate(divide="ignore"):
        good_k = min(1 - 1 / np.log10(S), 0.7)
    return {"elpd_loo": e.sum(), "se": np.sqrt(len(e) * e.var()), "p_loo": lppd.sum() - e.sum(), "lppd": lppd.sum(),
            "pointwise": e, "pareto_k": k, "good_k": good_k, "n_k_above_good": int((k > good_k).sum()),
            "n_k_above_0.7": int((k > 0.7).sum())}
