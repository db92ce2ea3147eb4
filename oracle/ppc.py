"""Restatement of the posterior predictive check kernel (``csrc/ppc.cu``) in float64 numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Definition (the same text as ``include/bplx.h``, ``csrc/ppc.cu`` and DESIGN §3f):

* Replicate ``n = (first_draw + s) * R + r`` (R = ``sims_per_draw``) uses posterior draw ``s``.  Its random numbers
  are ``curand_init(seed, n, 0)`` followed by ``curand()`` (Philox4_32_10).  Words ``2m`` and ``2m + 1`` become ``u_h``
  and ``u_a`` of observed match ``m`` through ``curand_uniform``: exactly the word addresses ``bplx_simulate_table``
  gives fixture ``f``.
* One match of one replicate is drawn by the season simulation's sampler, unchanged (``simulate.sample_scores``): the
  predict path's rates (neutral venues and confederations included, Extended's clip not applied); the draw's own grid up
  to ``max_goals``, with tau clamped at 0, normalised by its sum; inverse CDF over home goals, then over away goals given
  home goals.  A replicate that meets a non-finite rate or normaliser is invalid.  Match weights are ignored.
* Statistics per replicate (integers): ``score_counts [B, B]`` (matches with ``min(hg, B - 1) = i``,
  ``min(ag, B - 1) = j``), ``outcome_counts [3]`` (home wins, draws, away wins), ``goals [2]`` (home, away),
  ``total_goals_sq`` (``sum_m (hg + ag)^2``), ``team_points``, ``team_goals_for``, ``team_goals_against [T]`` per model
  team (``points = (win, draw)``).
* Posterior predictive p-value per element: the mid-p ``P(T_rep > T_obs) + 1/2 P(T_rep = T_obs)`` over the replicates.
"""
from __future__ import annotations

import numpy as np

from . import philox
from . import simulate as osim


def replicate(model, samples, observations, max_goals, sims_per_draw, seed, first_draw=0):
    """The replicated scores of the observed matches for the draws ``samples`` (the call's range; ``first_draw`` is the
    global index of its first draw): ``home`` / ``away`` / ``margin [N, M]`` (``simulate.sample_scores``'s margin) and
    ``valid [N]``; a match that makes its replicate invalid has scores 255."""
    M = len(observations["home_team"])
    words, s_of = osim.philox_words(samples, sims_per_draw, seed, first_draw, 2 * M)
    zeros = np.zeros(M, np.int64)  # (every match is on the one-slot "table" the simulation helper needs)
    return osim.play_fixtures(model, samples, observations, zeros, zeros, 1, max_goals, s_of,
                              philox.uniform(words).astype(np.float64))


def statistics(home_team, away_team, home, away, num_teams, score_bins=6, points=(3, 1)):
    """The statistics of given scores ``home`` / ``away [n, M]``, counted match by match: a dict of int64 arrays
    ``[n, ...]``."""
    home, away = np.atleast_2d(np.asarray(home, np.int64)), np.atleast_2d(np.asarray(away, np.int64))
    n, M = home.shape
    B, T = int(score_bins), int(num_teams)
    pw, pd = (int(x) for x in points)
    out = {"score_counts": np.zeros((n, B, B), np.int64), "outcome_counts": np.zeros((n, 3), np.int64),
           "goals": np.zeros((n, 2), np.int64), "total_goals_sq": np.zeros(n, np.int64),
           "team_points": np.zeros((n, T), np.int64), "team_goals_for": np.zeros((n, T), np.int64),
           "team_goals_against": np.zeros((n, T), np.int64)}
    rows = np.arange(n)
    for m in range(M):
        h, a = home[:, m], away[:, m]
        ht, at = int(home_team[m]), int(away_team[m])
        out["score_counts"][rows, np.minimum(h, B - 1), np.minimum(a, B - 1)] += 1
        out["outcome_counts"][rows, np.where(h > a, 0, np.where(h == a, 1, 2))] += 1
        out["goals"][:, 0] += h
        out["goals"][:, 1] += a
        out["total_goals_sq"] += (h + a) ** 2
        out["team_points"][:, ht] += np.where(h > a, pw, np.where(h == a, pd, 0))
        out["team_points"][:, at] += np.where(a > h, pw, np.where(h == a, pd, 0))
        out["team_goals_for"][:, ht] += h
        out["team_goals_against"][:, ht] += a
        out["team_goals_for"][:, at] += a
        out["team_goals_against"][:, at] += h
    return out


def mid_p(replicates, observed):
    """``P(T_rep > T_obs) + 1/2 P(T_rep = T_obs)`` per element, over the leading axis of ``replicates``."""
    rep = np.asarray(replicates, np.float64)
    obs = np.asarray(observed, np.float64)
    return np.mean(rep > obs, axis=0) + 0.5 * np.mean(rep == obs, axis=0)
