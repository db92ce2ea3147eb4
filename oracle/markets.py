"""Per-draw market probabilities: the float64 reference of ``bplx_market_draws``.

TEST INFRASTRUCTURE ONLY.  Definitions (the same in ``include/bplx.h`` and the predictor docstring): for posterior draw
s and fixture f the rates lh, la are ``oracle/predict.py``'s ``expected_goals`` (neutral venues and confederations, no
clip), c = corr_coef[s], G = max_goals, and the draw's grid is

    P_s(i, j) = tau(i, j) e^-lh lh^i / i! e^-la la^j / j!,   0 <= i, j <= G,

with tau clamped at 0 on the four low cells ((0,0) 1 - c lh la, (0,1) 1 + c lh, (1,0) 1 + c la, (1,1) 1 - c).  The
grid is not normalised.  Rows per fixture: home_win, draw, away_win (i > j, i = j, i < j), both_teams_score (i >= 1 and
j >= 1), home_rate, away_rate (lh, la), per total line L total_over_L (i + j > L) and total_under_L (i + j < L), per
margin line h home_margin_over_h (i - j > h) and home_margin_under_h (i - j < h).  Every row is a literal sum of the
cells of the full (G + 1) x (G + 1) grid: no separable shortcut.
"""
from __future__ import annotations

import numpy as np
from scipy.special import gammaln

from . import predict as op


def market_names(total_lines=(), margin_lines=()):
    names = ["home_win", "draw", "away_win", "both_teams_score", "home_rate", "away_rate"]
    for x in total_lines:
        names += [f"total_over_{float(x):g}", f"total_under_{float(x):g}"]
    for x in margin_lines:
        names += [f"home_margin_over_{float(x):g}", f"home_margin_under_{float(x):g}"]
    return names


def draw_grids(lh, la, corr_coef, max_goals):
    """``[S, F, g, g]`` float64 grids of the definition from ``[S, F]`` rates and ``[S]`` corr_coef."""
    lh, la = np.asarray(lh, np.float64), np.asarray(la, np.float64)
    c = np.asarray(corr_coef, np.float64)[:, None]
    k = np.arange(max_goals + 1, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        ph = np.exp(k * np.log(lh[..., None]) - lh[..., None] - gammaln(k + 1.0))
        pa = np.exp(k * np.log(la[..., None]) - la[..., None] - gammaln(k + 1.0))
    grid = ph[..., :, None] * pa[..., None, :]
    tau = np.ones(grid.shape)
    tau[..., 0, 0] = np.clip(1.0 - c * lh * la, 0.0, None)
    tau[..., 0, 1] = np.clip(1.0 + c * lh, 0.0, None)
    tau[..., 1, 0] = np.clip(1.0 + c * la, 0.0, None)
    tau[..., 1, 1] = np.clip(np.broadcast_to(1.0 - c, lh.shape), 0.0, None)
    return tau * grid


def market_masks(max_goals, total_lines=(), margin_lines=()):
    """``{row name: [g, g] bool}`` of the cells each probability row sums."""
    n = np.arange(max_goals + 1)
    i, j = np.meshgrid(n, n, indexing="ij")
    m = {"home_win": i > j, "draw": i == j, "away_win": i < j, "both_teams_score": (i >= 1) & (j >= 1)}
    for x in total_lines:
        m[f"total_over_{float(x):g}"] = i + j > x
        m[f"total_under_{float(x):g}"] = i + j < x
    for x in margin_lines:
        m[f"home_margin_over_{float(x):g}"] = i - j > x
        m[f"home_margin_under_{float(x):g}"] = i - j < x
    return m


def market_draws(model, samples, home, away, max_goals, total_lines=(), margin_lines=(), chunk=16, **fx):
    """``[S, F, K]`` float64 values of the K rows of ``market_names(total_lines, margin_lines)`` per draw and fixture
    (the grids are formed ``chunk`` fixtures at a time)."""
    lh, la = op.expected_goals(model, samples, home, away, **fx)
    masks = market_masks(max_goals, total_lines, margin_lines)
    names = market_names(total_lines, margin_lines)
    out = np.empty(lh.shape + (len(names),))
    for lo in range(0, lh.shape[1], chunk):
        sl = slice(lo, lo + chunk)
        grids = draw_grids(lh[:, sl], la[:, sl], samples["corr_coef"], max_goals)
        for k, name in enumerate(names):
            if name == "home_rate":
                out[:, sl, k] = lh[:, sl]
            elif name == "away_rate":
                out[:, sl, k] = la[:, sl]
            else:
                out[:, sl, k] = (grids * masks[name]).sum(axis=(-2, -1))
    return out
