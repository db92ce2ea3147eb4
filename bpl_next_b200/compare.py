"""Model comparison totals from per-match values: WAIC, PSIS-LOO and ``compare``.

The per-match values come from the CUDA kernels (``problem.pointwise_loglik`` and ``problem.psis_loo``); this module
only does the host arithmetic on ``[M]`` arrays, in float64.  Definitions, for S posterior draws and M matches with
pointwise log-likelihood ``ll[s, m]``:

* ``lppd_m = logsumexp_s ll - log S``
* ``p_waic_m = var_s ll`` with divisor S (ddof 0), ``elpd_waic_m = lppd_m - p_waic_m``
* ``elpd_loo_m``: PSIS-LOO of match m (ArviZ's ``_psislw``); ``elpd_loo = sum_m elpd_loo_m``,
  ``se = sqrt(M var0(elpd_loo_m))``, ``p_loo = sum_m lppd_m - elpd_loo``
* k-hat warnings: the count of ``k > min(1 - 1/log10 S, 0.7)`` and the count of ``k > 0.7``.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np


def lppd_from_stats(stats: np.ndarray, num_samples: int) -> np.ndarray:
    """``stats [M, 4]`` = (max ll, sum exp(ll - max), sum ll, sum ll^2) -> ``lppd_m [M]``."""
    st = np.asarray(stats, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return st[:, 0] + np.log(st[:, 1]) - np.log(num_samples)


def _se(x: np.ndarray) -> float:
    return float(np.sqrt(len(x) * np.var(x)))


def waic_from_stats(stats: np.ndarray, num_samples: int, match_key: Optional[str] = None) -> Dict:
    """WAIC totals from the pointwise kernel's statistics."""
    st = np.asarray(stats, dtype=np.float64)
    S = float(num_samples)
    lppd = lppd_from_stats(st, num_samples)
    mean = st[:, 2] / S
    with np.errstate(invalid="ignore"):
        p = np.maximum(st[:, 3] / S - mean * mean, 0.0)  # (a rounding-negative variance is 0)
    e = lppd - p
    return {"elpd_waic": float(e.sum()), "se": _se(e), "p_waic": float(p.sum()), "lppd": float(lppd.sum()),
            "pointwise": e, "lppd_pointwise": lppd, "p_waic_pointwise": p, "num_samples": int(num_samples),
            "num_matches": len(e), "match_key": match_key}


def loo_from_pointwise(elpd_i: np.ndarray, pareto_k: np.ndarray, lppd: np.ndarray, num_samples: int,
                       r_eff: float = 1.0, match_key: Optional[str] = None) -> Dict:
    """PSIS-LOO totals from the PSIS kernel's ``elpd_loo_m`` and ``k-hat`` and the pointwise ``lppd_m``."""
    e = np.asarray(elpd_i, dtype=np.float64)
    k = np.asarray(pareto_k, dtype=np.float64)
    lppd = np.asarray(lppd, dtype=np.float64)
    with np.errstate(divide="ignore"):
        good_k = min(1.0 - 1.0 / np.log10(num_samples), 0.7) if num_samples > 1 else -np.inf
    return {"elpd_loo": float(e.sum()), "se": _se(e), "p_loo": float(lppd.sum() - e.sum()), "lppd": float(lppd.sum()),
            "pointwise": e, "pareto_k": k, "good_k": float(good_k), "n_k_above_good": int((k > good_k).sum()),
            "n_k_above_0.7": int((k > 0.7).sum()), "r_eff": float(r_eff), "num_samples": int(num_samples),
            "num_matches": len(e), "match_key": match_key}


def compare(results: Dict[str, Dict]) -> Dict[str, Dict]:
    """Ranks ``loo()`` results of several fits by ``elpd_loo`` (best first).

    Returns ``{name: {"rank", "elpd_loo", "p_loo", "se", "d_elpd", "dse", "n_k_above_0.7"}}`` in rank order, where
    ``d_elpd = elpd_loo(best) - elpd_loo(name)`` and ``dse = sqrt(M var0(elpd_m(best) - elpd_m(name)))`` are taken
    match by match against the best model (both 0 for the best itself).  Results computed on different matches (a
    different ``match_key`` or number of matches) are refused: pointwise differences mean nothing across data sets.
    """
    if not results:
        raise ValueError("compare needs at least one result")
    for name, r in results.items():
        if "elpd_loo" not in r or "pointwise" not in r:
            raise ValueError(f"{name!r} is not a loo() result")
    items = list(results.items())
    key0, m0 = items[0][1].get("match_key"), len(items[0][1]["pointwise"])
    for name, r in items[1:]:
        if len(r["pointwise"]) != m0 or r.get("match_key") != key0:
            raise ValueError(f"{name!r} was computed on different matches than {items[0][0]!r}: cannot compare")
    ranked = sorted(items, key=lambda kv: -kv[1]["elpd_loo"])
    best = np.asarray(ranked[0][1]["pointwise"], dtype=np.float64)
    out = {}
    for rank, (name, r) in enumerate(ranked):
        diff = best - np.asarray(r["pointwise"], dtype=np.float64)
        out[name] = {"rank": rank, "elpd_loo": r["elpd_loo"], "p_loo": r["p_loo"], "se": r["se"],
                     "d_elpd": float(diff.sum()), "dse": _se(diff), "n_k_above_0.7": r["n_k_above_0.7"]}
    return out
