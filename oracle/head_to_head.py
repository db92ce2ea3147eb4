"""Restatement of the head-to-head ranking rule of season, group-stage and tournament simulation (``csrc/simulate.cu``,
``simulate_h2h_kernel``) in integer numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  It builds on ``oracle/simulate.py`` (same Philox words, same
score walks; its ``rank`` is the ``goal_difference`` rule) and ranks given scores.

Definition (the same text as ``include/bplx.h``): under ``head_to_head`` the teams of each group are ranked as follows.

1. Points.
2. Head-to-head among a level set.  For a set S of two or more teams level on points, each team's points, goal
   difference and goals for are computed over the matches between teams of S only: the played matches (``played_h2h``)
   and this simulation's simulated fixtures.  S is ordered by (head-to-head points, head-to-head goal difference,
   head-to-head goals for), all descending.
3. Reapply to what is still level.  If step 2 splits S, any part of two or more teams still level on all three values
   goes through step 2 again, with S being that part: only the matches among that part count.
4. Fall back when nobody separates.  A set in which step 2 separates nobody is ordered by overall goal difference,
   overall goals for, the tie-break key (word ``2F + t``), then the lower slot.

Position k is the team's index in this order.  Best-placed qualifiers are still ranked across groups by points, goal
difference, goals for and the key (``oracle.tournament.qualifiers``).  ``played_h2h [T, T, 2]`` holds the points and
goals of slot u against slot v in played matches.
"""
from __future__ import annotations

import numpy as np

from oracle import simulate as osim

RULES = ("goal_difference", "head_to_head")


def order_level_set(level, pair, gd, gf, keys):
    """Steps 2-4 for one set ``level`` (slots level on points) of one simulation: the slots in ranking order.
    ``pair [T, T, 2]``: points and goals of u against v over the played and simulated matches; ``gd``, ``gf``,
    ``keys [T]`` the overall values."""
    level = list(level)
    if len(level) < 2:
        return level

    def h2h(x):
        ys = [y for y in level if y != x]
        return (int(pair[x, ys, 0].sum()), int(pair[x, ys, 1].sum() - pair[ys, x, 1].sum()), int(pair[x, ys, 1].sum()))

    tri = {x: h2h(x) for x in level}
    if len(set(tri.values())) == 1:  # nobody separated: overall goal difference, goals for, the key, the lower slot
        return sorted(level, key=lambda x: (-gd[x], -gf[x], -keys[x], x))
    out = []
    for v in sorted(set(tri.values()), reverse=True):
        out += order_level_set([x for x in level if tri[x] == v], pair, gd, gf, keys)
    return out


def pair_results(table, home_slot, away_slot, home, away, played_h2h=None):
    """``[T, T, 2]`` of one simulation: points and goals of u against v in ``played_h2h`` plus the fixtures with scores
    ``home`` / ``away [F]``."""
    T = len(table["start_points"])
    pw, pd = int(table["points_win"]), int(table["points_draw"])
    pair = np.zeros((T, T, 2), np.int64) if played_h2h is None else np.array(played_h2h, np.int64)
    for u, v, x, y in zip(home_slot, away_slot, home, away):
        pair[u, v] += (pw if x > y else pd if x == y else 0, x)
        pair[v, u] += (pw if y > x else pd if x == y else 0, y)
    return pair


def rank(table, home_slot, away_slot, home, away, keys, played_h2h=None, tiebreak="head_to_head"):
    """Positions ``[n, T]`` (0-based, within the group) of scores ``home`` / ``away [n, F]`` with tie-break keys
    ``[n, T]`` under ``tiebreak``; ``goal_difference`` is ``oracle.simulate.rank``."""
    if tiebreak not in RULES:
        raise ValueError(f"unknown tiebreak {tiebreak!r}")
    hs, as_ = np.asarray(home_slot, np.int64), np.asarray(away_slot, np.int64)
    home, away, keys = (np.asarray(x, np.int64) for x in (home, away, keys))
    pts, gd, gf = osim.tables(table, hs, as_, home, away)
    if tiebreak == "goal_difference":
        return osim.rank(pts, gd, gf, keys, table.get("group"))
    n, T = pts.shape
    group = np.zeros(T, np.int64) if table.get("group") is None else np.asarray(table["group"], np.int64)
    members = [np.flatnonzero(group == g) for g in np.unique(group)]
    out = np.empty((n, T), np.int64)
    for i in range(n):
        pair = None
        for mem in members:
            by_pts = sorted(mem, key=lambda x: -pts[i, x])
            order, p = [], 0
            while p < len(by_pts):
                q = p
                while q < len(by_pts) and pts[i, by_pts[q]] == pts[i, by_pts[p]]:
                    q += 1
                if q - p > 1 and pair is None:
                    pair = pair_results(table, hs, as_, home[i], away[i], played_h2h)
                order += by_pts[p:q] if q - p == 1 else order_level_set(by_pts[p:q], pair, gd[i], gf[i], keys[i])
                p = q
            out[i, order] = np.arange(len(order))
    return out


def rank_scores(table, home_slot, away_slot, home, away, keys, valid=None, tiebreak="head_to_head", played_h2h=None):
    """``oracle.simulate.rank_scores`` under ``tiebreak``: ``positions [n, T]`` (255 for invalid simulations),
    ``position_counts [T, P]``, ``points_counts [T, B]``."""
    n = np.asarray(home).shape[0]
    valid = np.ones(n, bool) if valid is None else np.asarray(valid, bool)
    hv, av = np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0)
    pts, _, _ = osim.tables(table, home_slot, away_slot, hv, av)
    pos = rank(table, home_slot, away_slot, hv, av, keys, played_h2h, tiebreak)
    return osim.histograms(table, pts, pos, valid)


def simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed, first_draw=0,
             tiebreak="head_to_head", played_h2h=None):
    """``oracle.simulate.simulate`` with the groups ranked under ``tiebreak``: the same scores, keys, margins and
    validity (the rule reads no other Philox word), then ``rank_scores``'s outputs."""
    out = osim.simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed,
                        first_draw)
    T = len(table["start_points"])
    hs, as_ = (np.minimum(np.asarray(x, np.int64), T - 1) for x in (home_slot, away_slot))
    out.update(rank_scores(table, hs, as_, out["home"], out["away"], out["keys"], out["valid"], tiebreak, played_h2h))
    return out
