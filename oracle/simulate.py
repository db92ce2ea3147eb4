"""Restatement of the season / group-stage simulation (``csrc/simulate.cu``) in float64 numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Definition (the same text as ``include/bplx.h`` and ``csrc/simulate.cu``):

* Simulation ``n = (first_draw + s) * R + r`` uses draw ``s``.  Its random numbers are the outputs of
  ``curand_init(seed, n, 0)`` followed by ``curand()`` (Philox4_32_10, ``philox.stream(seed, n, 0, 2F + T_tab)``).
  Words ``2f`` and ``2f + 1`` are ``u_h`` and ``u_a`` of fixture ``f`` through ``curand_uniform`` (in (0, 1]); word
  ``2F + t`` is the tie-break key of table slot ``t``.
* Fixture ``f`` in draw ``s``: ``lambda_h``, ``lambda_a`` are the predict path's rates (``predict.expected_goals``);
  ``w(i, j) = tau+(i, j) Pois(i; lambda_h) Pois(j; lambda_a)`` for ``0 <= i, j <= G`` with ``tau+`` = tau clamped at 0
  (``predict.correlation_term``'s four cells) and 1 elsewhere; ``Z = sum w``, ``m(i) = sum_j w(i, j)``.  Home goals are
  the smallest ``i`` with ``sum_{i' <= i} m(i') >= u_h Z``, away goals the smallest ``j`` with
  ``sum_{j' <= j} w(i, j') >= u_a m(i)``; when no index meets a target, the last index with positive mass.  A cell of
  zero probability is never returned.  The weights are taken un-normalised (``lambda^k / k!``): ``e^-lambda`` cancels.
  A fixture with a non-finite rate or a normaliser that is not positive and finite makes the simulation invalid (its
  scores are 255, its positions row 255, and it is left out of the histograms).
* Table: ``points_win`` / ``points_draw``; teams ranked within their group by points, goal difference, goals for, then
  the tie-break key, all descending, then the lower slot.  Position = the number of teams of the group ranked ahead.
  Head-to-head and fair-play rules are not modelled: ties left after goals for are decided by lot.

``margin`` of a (simulation, fixture): the smallest distance of ``u_h Z`` from a cumulative boundary of the home walk,
relative to ``Z``, and of ``u_a m(i)`` from one of the away walk, relative to ``m(i)`` -- the float32 kernel may pick a
neighbouring cell only where this is at rounding level.
"""
from __future__ import annotations

import numpy as np

from . import philox
from . import predict as op

_CHUNK = 8192  # simulations per block of the [n, g, g] weights


def _pmf_unnormalised(lam, G):
    """``lam^k / k!`` for ``k = 0 .. G``, ``[n, G + 1]`` (the recurrence ``p_k = p_{k-1} lam / k``)."""
    with np.errstate(over="ignore", invalid="ignore"):
        steps = lam[:, None] / np.arange(1, G + 1, dtype=np.float64)[None, :]
        return np.concatenate([np.ones((len(lam), 1)), np.cumprod(steps, axis=1)], axis=1)


def _walk(mass, u):
    """Smallest index whose cumulative mass reaches ``u * total`` among indices of positive mass, else the last index of
    positive mass; and the relative distance of the target from the nearest cumulative boundary."""
    cum = np.cumsum(mass, axis=1)
    total = cum[:, -1]
    target = u * total
    pos = mass > 0
    hit = (cum >= target[:, None]) & pos
    last = mass.shape[1] - 1 - np.argmax(pos[:, ::-1], axis=1)
    idx = np.where(hit.any(axis=1), np.argmax(hit, axis=1), last)
    with np.errstate(invalid="ignore", divide="ignore"):
        margin = np.abs(target[:, None] - cum).min(axis=1) / total
    return idx, margin


def sample_scores(lh, la, c, uh, ua, max_goals):
    """Scores of one fixture for ``n`` simulations: rates / corr_coef / uniforms ``[n]`` (float64; the uniforms are the
    kernel's float32 values).  Returns ``(home, away, margin, valid)``; invalid entries have scores 255."""
    G = int(max_goals)
    n = len(lh)
    home = np.full(n, 255, np.int64)
    away = np.full(n, 255, np.int64)
    margin = np.full(n, np.inf)
    valid = np.zeros(n, bool)
    for lo in range(0, n, _CHUNK):
        sl = slice(lo, min(n, lo + _CHUNK))
        h_, a_, c_ = lh[sl], la[sl], c[sl]
        p, q = _pmf_unnormalised(h_, G), _pmf_unnormalised(a_, G)
        with np.errstate(over="ignore", invalid="ignore"):
            w = p[:, :, None] * q[:, None, :]
            w[:, 0, 0] *= np.maximum(1.0 - c_ * h_ * a_, 0.0)
            w[:, 0, 1] *= np.maximum(1.0 + c_ * h_, 0.0)
            w[:, 1, 0] *= np.maximum(1.0 + c_ * a_, 0.0)
            w[:, 1, 1] *= np.maximum(1.0 - c_, 0.0)
            m = w.sum(axis=2)
            Z = m.sum(axis=1)
        ok = np.isfinite(h_) & np.isfinite(a_) & np.isfinite(Z) & (Z > 0)
        if not ok.any():
            continue
        i, mh = _walk(m[ok], uh[sl][ok])
        row = w[ok][np.arange(ok.sum()), i]
        j, ma = _walk(row, ua[sl][ok])
        idx = np.arange(sl.start, sl.stop)[ok]
        home[idx], away[idx], margin[idx], valid[idx] = i, j, np.minimum(mh, ma), True
    return home, away, margin, valid


def rank(points, goal_diff, goals_for, keys, group=None):
    """Positions ``[n, T]`` (0-based, within the group) from final tables ``[n, T]`` (integers) and tie-break keys."""
    points, goal_diff, goals_for = (np.asarray(x, np.int64) for x in (points, goal_diff, goals_for))
    keys = np.asarray(keys, np.int64)
    n, T = points.shape
    g = np.zeros(T, np.int64) if group is None else np.asarray(group, np.int64)
    same = g[:, None] == g[None, :]  # [t, u]
    u_lt_t = np.arange(T)[None, :] < np.arange(T)[:, None]
    out = np.empty((n, T), np.int64)
    for lo in range(0, n, _CHUNK):
        sl = slice(lo, min(n, lo + _CHUNK))
        ahead = np.broadcast_to(u_lt_t, (sl.stop - sl.start, T, T))
        for x in (keys, goals_for, goal_diff, points):  # innermost criterion first
            a = x[sl]
            gt, eq = a[:, None, :] > a[:, :, None], a[:, None, :] == a[:, :, None]  # [n, t, u]: u's value vs t's
            ahead = gt | (eq & ahead)
        out[sl] = (ahead & same[None]).sum(axis=2)
    return out


def tables(table, home_slot, away_slot, home, away):
    """Final points, goal difference and goals for ``[n, T]`` of the simulations with scores ``home`` / ``away``
    ``[n, F]`` (valid simulations only are meaningful)."""
    T = len(table["start_points"])
    hs, as_ = np.asarray(home_slot, np.int64), np.asarray(away_slot, np.int64)
    home, away = np.asarray(home, np.int64), np.asarray(away, np.int64)
    n = home.shape[0]
    pw, pd = int(table["points_win"]), int(table["points_draw"])
    ph = np.where(home > away, pw, np.where(home == away, pd, 0))
    pa = np.where(away > home, pw, np.where(home == away, pd, 0))
    pts = np.tile(np.asarray(table["start_points"], np.int64), (n, 1))
    gf = np.tile(np.asarray(table["start_goals_for"], np.int64), (n, 1))
    ga = np.tile(np.asarray(table["start_goals_against"], np.int64), (n, 1))
    rows = np.arange(n)[:, None]
    for arr, sl, v in ((pts, hs, ph), (pts, as_, pa), (gf, hs, home), (gf, as_, away), (ga, hs, away), (ga, as_, home)):
        np.add.at(arr, (np.broadcast_to(rows, v.shape), np.broadcast_to(sl[None, :], v.shape)), v)
    return pts, gf - ga, gf


def rank_scores(table, home_slot, away_slot, home, away, keys, valid=None):
    """The ranking and histograms of given scores ``[n, F]`` with tie-break keys ``[n, T]``: ``positions [n, T]``
    (255 for invalid simulations), ``position_counts [T, P]``, ``points_counts [T, B]`` (gained points)."""
    n = np.asarray(home).shape[0]
    valid = np.ones(n, bool) if valid is None else np.asarray(valid, bool)
    pts, gd, gf = tables(table, home_slot, away_slot, np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0))
    return histograms(table, pts, rank(pts, gd, gf, keys, table.get("group")), valid)


def histograms(table, pts, pos, valid):
    """``rank_scores``'s outputs from final points and positions ``[n, T]``, counting the simulations ``valid [n]``."""
    T = len(table["start_points"])
    P, B = int(table["num_positions"]), int(table["num_points_bins"])
    pc = np.zeros((T, P), np.int64)
    bc = np.zeros((T, B), np.int64)
    gained = pts - np.asarray(table["start_points"], np.int64)[None, :]
    cols = np.broadcast_to(np.arange(T)[None, :], pos.shape)
    np.add.at(pc, (cols[valid], pos[valid]), 1)
    np.add.at(bc, (cols[valid], gained[valid]), 1)
    pos = np.where(valid[:, None], pos, 255)
    return {"positions": pos, "position_counts": pc, "points_counts": bc}


def philox_words(samples, sims_per_draw, seed, first_draw, count):
    """Words ``0 .. count - 1`` of every simulation ``n = (first_draw + s) R + r`` (draw-major), ``[S R, count]``, and
    the draw ``s`` of each simulation ``[S R]``."""
    S, R = np.asarray(samples["attack"]).shape[0], int(sims_per_draw)
    s_of = np.repeat(np.arange(S), R)
    n_glob = (first_draw + s_of) * R + np.tile(np.arange(R), S)
    return philox.stream(int(seed), n_glob.astype(np.uint64), 0, count), s_of


def play_fixtures(model, samples, fixtures, home_slot, away_slot, T, max_goals, s_of, u):
    """The fixtures of simulations of draws ``s_of [N]`` with uniforms ``u [N, 2F]`` (words ``2f``, ``2f + 1``):
    ``home`` / ``away`` / ``margin [N, F]`` and ``valid [N]``; a fixture that makes its simulation invalid (a slot
    outside the table of ``T`` slots included) has scores 255."""
    kw = {k: fixtures[k] for k in ("home_conf", "away_conf", "neutral_venue") if fixtures.get(k) is not None}
    if model in ("neutral", "neutral_wc") and "neutral_venue" not in kw:
        kw["neutral_venue"] = np.zeros(len(fixtures["home_team"]), np.uint8)
    with np.errstate(over="ignore", invalid="ignore"):
        lh, la = op.expected_goals(model, samples, fixtures["home_team"], fixtures["away_team"], **kw)  # [S, F]
    cc = np.asarray(samples["corr_coef"], np.float64)
    N, F = len(s_of), lh.shape[1]
    home = np.empty((N, F), np.int64)
    away = np.empty((N, F), np.int64)
    margin = np.empty((N, F))
    valid = np.ones(N, bool)
    hs, as_ = np.asarray(home_slot, np.int64), np.asarray(away_slot, np.int64)
    for f in range(F):
        h, a, m, v = sample_scores(lh[s_of, f], la[s_of, f], cc[s_of], u[:, 2 * f], u[:, 2 * f + 1], max_goals)
        v &= (hs[f] < T) & (as_[f] < T)
        home[:, f], away[:, f], margin[:, f] = np.where(v, h, 255), np.where(v, a, 255), m
        valid &= v
    return home, away, margin, valid


def simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed, first_draw=0):
    """The simulations of draws ``samples`` (the call's range; ``first_draw`` is the global index of its first draw).
    Returns ``home`` / ``away`` / ``margin`` ``[N, F]``, ``keys [N, T]``, ``valid [N]``, and ``rank_scores``'s
    ``positions``, ``position_counts``, ``points_counts``, with ``invalid`` = the number of invalid simulations."""
    F, T = len(fixtures["home_team"]), len(table["start_points"])
    words, s_of = philox_words(samples, sims_per_draw, seed, first_draw, 2 * F + T)  # [N, 2F + T]
    home, away, margin, valid = play_fixtures(model, samples, fixtures, home_slot, away_slot, T, max_goals, s_of,
                                              philox.uniform(words[:, :2 * F]).astype(np.float64))
    keys = words[:, 2 * F:].astype(np.int64)
    hs, as_ = np.minimum(np.asarray(home_slot, np.int64), T - 1), np.minimum(np.asarray(away_slot, np.int64), T - 1)
    out = rank_scores(table, hs, as_, home, away, keys, valid)
    out.update(home=home, away=away, margin=margin, keys=keys, valid=valid, invalid=int((~valid).sum()))
    return out
