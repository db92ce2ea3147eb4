"""Host summary of posterior predictive checks (``_BplxPredictor.posterior_predictive_check``): the statistics of the
observed scores, and the mean, standard deviation and posterior predictive p-value of every statistic over the
replicates that ``bplx_posterior_predictive`` computes on the GPU.  numpy only: no device is needed here.

Statistics of a set of scores of M matches (the same definitions as ``include/bplx.h`` and ``oracle/ppc.py``):

* ``score_counts [B, B]``: matches with ``min(hg, B - 1) = i``, ``min(ag, B - 1) = j`` (B = ``score_bins``);
* ``outcome_counts [3]``: home wins, draws, away wins ("home" = the listed home team, neutral venue or not);
* ``goals [2]``: total home goals, total away goals;
* ``total_goals_sq []``: ``sum_m (hg + ag)^2``;
* ``team_points``, ``team_goals_for``, ``team_goals_against [T]``: per model team, ``points = (win, draw)``;
* ``total_goals_dispersion []``: variance over mean of the total goals per match, from ``goals`` and
  ``total_goals_sq``.

Posterior predictive p-value per element: the mid-p ``P(T_rep > T_obs) + 1/2 P(T_rep = T_obs)`` over the N
replicates.  Near 0.5 the data sit inside what the model predicts; near 0 or 1 the model misses.  A team with no
matches gets 0.5 (every replicate equals the observed 0).
"""
from __future__ import annotations

from typing import Dict

import numpy as np

# the statistics the device computes per replicate, in the order of bplx_ppc_output
STATISTICS = ("score_counts", "outcome_counts", "goals", "total_goals_sq", "team_points", "team_goals_for",
              "team_goals_against")


def statistics(home_team, away_team, home_goals, away_goals, num_teams: int, score_bins: int = 6,
               points=(3, 1)) -> Dict[str, np.ndarray]:
    """The statistics of one set of scores of M matches (int64; goals above any ``max_goals`` count as they are)."""
    ht, at = np.asarray(home_team, np.int64), np.asarray(away_team, np.int64)
    hg, ag = np.asarray(home_goals, np.int64), np.asarray(away_goals, np.int64)
    B, T = int(score_bins), int(num_teams)
    pw, pd = (int(x) for x in points)
    cells = np.bincount(np.minimum(hg, B - 1) * B + np.minimum(ag, B - 1), minlength=B * B).reshape(B, B)
    ph = np.where(hg > ag, pw, np.where(hg == ag, pd, 0))
    pa = np.where(ag > hg, pw, np.where(hg == ag, pd, 0))

    def per_team(home_value, away_value):
        out = np.zeros(T, np.int64)
        np.add.at(out, ht, home_value)
        np.add.at(out, at, away_value)
        return out

    return {"score_counts": cells.astype(np.int64),
            "outcome_counts": np.array([(hg > ag).sum(), (hg == ag).sum(), (hg < ag).sum()], np.int64),
            "goals": np.array([hg.sum(), ag.sum()], np.int64),
            "total_goals_sq": np.int64(((hg + ag) ** 2).sum()),
            "team_points": per_team(ph, pa), "team_goals_for": per_team(hg, ag), "team_goals_against": per_team(ag, hg)}


def dispersion(goals, total_goals_sq, num_matches: int) -> np.ndarray:
    """Variance over mean of the total goals per match, from ``goals [..., 2]`` and ``total_goals_sq [...]``: 1 for
    Poisson totals, above 1 for over-dispersed ones (NaN when no goal was scored)."""
    M = float(num_matches)
    mean = np.asarray(goals, np.float64).sum(axis=-1) / M
    var = np.asarray(total_goals_sq, np.float64) / M - mean ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        return var / mean


def mid_p(replicates, observed) -> np.ndarray:
    """``P(T_rep > T_obs) + 1/2 P(T_rep = T_obs)`` per element over the leading axis of ``replicates [N, ...]``."""
    rep, obs = np.asarray(replicates), np.asarray(observed)
    return ((rep > obs).sum(axis=0) + 0.5 * (rep == obs).sum(axis=0)) / rep.shape[0]


def summarize(observed: Dict[str, np.ndarray], replicates: Dict[str, np.ndarray],
              num_matches: int) -> Dict[str, Dict[str, np.ndarray]]:
    """Per statistic of ``STATISTICS`` and ``total_goals_dispersion``: ``observed``, ``mean`` and ``sd`` (over the
    replicates, divisor N) and ``p_value`` (``mid_p``)."""
    obs, rep = dict(observed), dict(replicates)
    obs["total_goals_dispersion"] = dispersion(obs["goals"], obs["total_goals_sq"], num_matches)
    rep["total_goals_dispersion"] = dispersion(rep["goals"], rep["total_goals_sq"], num_matches)
    out = {}
    for k in STATISTICS + ("total_goals_dispersion",):
        r = np.asarray(rep[k], np.float64)
        out[k] = {"observed": obs[k], "mean": r.mean(axis=0), "sd": r.std(axis=0), "p_value": mid_p(rep[k], obs[k])}
    return out
