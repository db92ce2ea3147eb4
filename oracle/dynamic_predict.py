"""Float64 restatement of the dynamic model's predictive distribution (``csrc/dynamic_predict.cu`` and the gameweek
calls of ``csrc/loo.cu`` / ``csrc/ppc.cu``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Definition (the same text as ``include/bplx.h``, ``csrc/dynamic_predict.cu``, DESIGN §3h and the docstrings):

* Only fits of the intended walk have a predictive distribution.  Gameweeks are 0-based, G = max + 1 as in ``fit``.
* Fitted gameweek (g < G): per draw, ``attack[g]``, ``defence[g]``, the four venue effects at g and ``corr_coef``; the
  rates are the NEUTRAL model's (``predict.expected_goals``), which are ``_model``'s at gameweek g.
* Forecast gameweek (g >= G): for each draw and gameweek j = G .. g in order, fresh sites from their priors --
  ``mean_home_attack``, ``mean_home_defence`` ~ N(0.1, 0.2), ``mean_away_attack``, ``mean_away_defence`` ~ N(-0.1, 0.2),
  the six ``std_*`` ~ HalfNormal(1), per team ``u`` ~ Beta(2, 4), ``rho = 2u - 1``, ``za`` ~ N(0, 1),
  ``zd = rho za + sqrt(1 - rho^2) eps``, the four ``*_decentered`` ~ N(0, 1) -- then
  ``attack[j] = attack[j - 1] + za std_attack[j]`` (defence with zd) and ``effect[j] = mean[j] + std[j] dec[j]``.
* Random numbers: Philox4_32_10 under the key ``seed ^ BPLX_FORECAST_KEY``, subsequence ``first_draw + s``; gameweek
  ``k = j - G`` uses counter blocks ``k P + 0 .. 2`` (P = 3 + 3T) for the draw and ``k P + 3 + 3t + 0 .. 2`` for team t
  (word map in ``include/bplx.h``).  The uniforms are the device's float32 values; the normals are float64 from them.
"""
from __future__ import annotations

import numpy as np

from . import philox
from . import ppc as oppc
from . import psis as opsis
from . import simulate as osim
from .models import layout_offsets, site_layout, standardise_covariates

FORECAST_KEY = 0x9E3779B97F4A7C15  # BPLX_FORECAST_KEY
EFFECTS = ("home_attack", "away_attack", "home_defence", "away_defence")
SITES = ("attack", "defence") + EFFECTS


def fitted_sites(theta, num_teams, num_gameweeks, covariates=None):
    """The sites ``fit`` records, from unconstrained draws ``theta [S, D]`` of the intended walk, in float64:
    ``attack`` / ``defence`` and the four venue effects ``[S, G, T]``."""
    theta = np.asarray(theta, np.float64)
    T, G = int(num_teams), int(num_gameweeks)
    K = 0 if covariates is None else int(np.asarray(covariates).shape[1])
    x = {}
    for name, (off, shape, tr) in layout_offsets(site_layout("dynamic", T, K, 0, G)).items():
        if name == "__D__":
            continue
        n = int(np.prod(shape)) if shape else 1
        v = theta[:, off:off + n]
        if tr == "exp":
            v = np.exp(v)
        elif tr == "sigmoid":
            v = 1.0 / (1.0 + np.exp(-v))
        x[name] = v.reshape((len(theta),) + tuple(shape)) if shape else v[:, 0]
    S = len(theta)
    a_mean, d_mean = np.zeros((S, T)), np.repeat(x["mean_defence"][:, None], T, axis=1)
    if K:
        Xs = np.asarray(standardise_covariates(np.asarray(covariates, np.float64)), np.float64)
        a_mean = x["attack_coefficients"] @ Xs.T
        d_mean = d_mean + x["defence_coefficients"] @ Xs.T
    out = {"attack": a_mean[:, None, :] + np.cumsum(x["standardised_attack"] * x["std_attack"][:, :, None], axis=1),
           "defence": d_mean[:, None, :] + np.cumsum(x["standardised_defence"] * x["std_defence"][:, :, None], axis=1)}
    for nm in EFFECTS:
        out[nm] = x["mean_" + nm][:, :, None] + x["std_" + nm][:, :, None] * x[nm + "_decentered"]
    return out


def slab(sites, g, corr_coef):
    """The NEUTRAL sample set of fitted gameweek ``g``: ``[S, T]`` sites and ``corr_coef [S]`` (float64)."""
    d = {k: np.asarray(sites[k], np.float64)[:, g] for k in SITES}
    d["corr_coef"] = np.asarray(corr_coef, np.float64)
    return d


def forecast_words(seed, num_teams, horizon, first_draw, num_draws):
    """The Philox words of the forecast, ``[S, horizon, 3 + 3T, 4]`` uint32 (block-major, as in include/bplx.h)."""
    T, h = int(num_teams), int(horizon)
    P = 3 + 3 * T
    key = (int(seed) ^ FORECAST_KEY) & 0xFFFFFFFFFFFFFFFF
    sub = (int(first_draw) + np.arange(int(num_draws))).astype(np.uint64)
    w = philox.stream(key, sub, 0, 4 * P * h)  # [S, 4 P h]
    return w.reshape(len(sub), h, P, 4)


def forecast_variates(words):
    """The variates of ``forecast_words``: per (draw, gameweek) ``mean_* [S, h]``, ``std_* [S, h]``; per team ``u``,
    ``za``, ``eps`` and the four ``*_decentered [S, h, T]`` (float64; u is the device's float32 value)."""
    wd, wt = words[:, :, :3, :].reshape(words.shape[0], words.shape[1], 12), words[:, :, 3:, :]
    T = wt.shape[2] // 3
    wt = wt.reshape(words.shape[0], words.shape[1], T, 12)
    v = {}
    n0, n1 = philox.box_muller(wd[..., 0], wd[..., 1])
    v["mean_home_attack"], v["mean_away_attack"] = 0.1 + 0.2 * n0, -0.1 + 0.2 * n1
    n0, n1 = philox.box_muller(wd[..., 2], wd[..., 3])
    v["mean_home_defence"], v["mean_away_defence"] = 0.1 + 0.2 * n0, -0.1 + 0.2 * n1
    n0, n1 = philox.box_muller(wd[..., 4], wd[..., 5])
    v["std_home_attack"], v["std_away_attack"] = np.abs(n0), np.abs(n1)
    n0, n1 = philox.box_muller(wd[..., 6], wd[..., 7])
    v["std_home_defence"], v["std_away_defence"] = np.abs(n0), np.abs(n1)
    n0, n1 = philox.box_muller(wd[..., 8], wd[..., 9])
    v["std_attack"], v["std_defence"] = np.abs(n0), np.abs(n1)
    u = np.sort(philox.uniform(wt[..., 0:5]), axis=-1)[..., 1]  # the 2nd smallest of 5: Beta(2, 4)
    v["u"] = u.astype(np.float64)
    v["za"], v["eps"] = philox.box_muller(wt[..., 6], wt[..., 7])
    v["home_attack_decentered"], v["away_attack_decentered"] = philox.box_muller(wt[..., 8], wt[..., 9])
    v["home_defence_decentered"], v["away_defence_decentered"] = philox.box_muller(wt[..., 10], wt[..., 11])
    return v


def forecast(attack_last, defence_last, horizon, seed, first_draw=0):
    """The forecast sites ``[horizon, S, T]`` (float64) from the walk at G - 1, replayed on the kernel's words."""
    att, dfn = np.asarray(attack_last, np.float64), np.asarray(defence_last, np.float64)
    S, T = att.shape
    v = forecast_variates(forecast_words(seed, T, horizon, first_draw, S))
    rho = 2.0 * v["u"] - 1.0
    zd = rho * v["za"] + np.sqrt(1.0 - rho ** 2) * v["eps"]
    out = {k: np.empty((int(horizon), S, T)) for k in SITES}
    for k in range(int(horizon)):
        att = att + v["za"][:, k] * v["std_attack"][:, k, None]
        dfn = dfn + zd[:, k] * v["std_defence"][:, k, None]
        out["attack"][k], out["defence"][k] = att, dfn
        for nm in EFFECTS:
            out[nm][k] = v["mean_" + nm][:, k, None] + v["std_" + nm][:, k, None] * v[nm + "_decentered"][:, k]
    return out


def pointwise_loglik(slabs, gameweek, home, away, home_goals, away_goals, neutral_venue):
    """``[S, M]`` float64 log-likelihood, match m under the NEUTRAL sample set ``slabs[gameweek[m]]``
    (``psis.pointwise_loglik`` per gameweek)."""
    gw = np.asarray(gameweek)
    S = len(slabs[int(gw[0])]["corr_coef"])
    out = np.empty((S, len(gw)))
    for g in np.unique(gw):
        m = gw == g
        out[:, m] = opsis.pointwise_loglik("neutral", slabs[int(g)], np.asarray(home)[m], np.asarray(away)[m],
                                           np.asarray(home_goals)[m], np.asarray(away_goals)[m],
                                           neutral_venue=np.asarray(neutral_venue)[m])
    return out


def replicate(slabs, gameweek, observations, max_goals, sims_per_draw, seed, first_draw=0):
    """``ppc.replicate`` with match m sampled from ``slabs[gameweek[m]]``: the same replicate index and words
    (2m, 2m + 1).  Returns ``home`` / ``away`` / ``margin [N, M]`` and ``valid [N]``."""
    gw = np.asarray(gameweek)
    M = len(gw)
    first = slabs[int(gw[0])]
    words, s_of = osim.philox_words(first, sims_per_draw, seed, first_draw, 2 * M)
    u = philox.uniform(words).astype(np.float64)
    N = len(s_of)
    home, away = np.empty((N, M), np.int64), np.empty((N, M), np.int64)
    margin, valid = np.empty((N, M)), np.ones(N, bool)
    for g in np.unique(gw):
        m = np.flatnonzero(gw == g)
        obs = {k: np.asarray(v)[m] for k, v in observations.items()}
        cols = np.stack([2 * m, 2 * m + 1], axis=1).ravel()
        zeros = np.zeros(len(m), np.int64)
        h, a, mg, v = osim.play_fixtures("neutral", slabs[int(g)], obs, zeros, zeros, 1, max_goals, s_of, u[:, cols])
        home[:, m], away[:, m], margin[:, m] = h, a, mg
        valid &= v
    return home, away, margin, valid


statistics = oppc.statistics
