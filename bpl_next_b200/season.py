"""Host arithmetic of season and group-stage simulation: the table, slots and groups in, probabilities out.

The simulation itself is the CUDA kernel behind ``problem.simulate_table`` (``csrc/simulate.cu``); this module builds its
inputs from team names and played results and turns its integer counts into probabilities.  Definition, in short (the
full text is in ``include/bplx.h``): every simulated season takes ONE posterior draw and plays every remaining fixture
with that draw's rates, so a team that is stronger in a draw is stronger in all of its matches of that season.  Teams
are ranked within their group by points, goal difference, goals for, then a random tie-break key; head-to-head and
fair-play rules are not modelled, so ties left after goals for are decided by lot.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Sequence, Tuple

import numpy as np

SIM_MAX_TEAMS = 64  # BPLX_SIM_MAX_TEAMS


def _names(x) -> list:
    return [x] if isinstance(x, (str, int, np.integer)) else list(x)


def table_teams(home, away, played: Optional[Dict[str, Any]] = None, teams=None) -> list:
    """The table: ``teams`` as given, or by default the sorted union of the teams in the fixtures and in ``played``."""
    if teams is not None:
        teams = list(teams)
        if len(set(teams)) != len(teams):
            raise ValueError("teams lists a team more than once")
        return teams
    names = set(_names(home)) | set(_names(away))
    if played is not None:
        names |= set(_names(played["home_team"])) | set(_names(played["away_team"]))
    return sorted(names)


def check_points(points) -> Tuple[int, int]:
    try:
        pw, pd = points
    except (TypeError, ValueError):
        raise ValueError(f"points must be a pair (win, draw), got {points!r}") from None
    if not all(isinstance(p, (int, np.integer)) and not isinstance(p, bool) for p in (pw, pd)):
        raise ValueError(f"points must be integers, got {points!r}")
    if not (pw >= 1 and 0 <= pd <= pw):
        raise ValueError(f"points must satisfy 0 <= draw <= win and win >= 1, got {points!r}")
    return int(pw), int(pd)


def build_table(teams: Sequence, played: Optional[Dict[str, Any]] = None, groups=None, points=(3, 1)) -> Dict[str, Any]:
    """Starting table of ``teams`` from ``played`` results (reference ``training_data`` keys: ``home_team``,
    ``away_team``, ``home_goals``, ``away_goals``): points (``points = (win, draw)``), goals for and against.  ``groups``
    is a mapping team -> label or a sequence of labels aligned with ``teams`` (None: one table); labels become ids
    0 .. K-1 in sorted order.  Returns the host table ``problem.simulate_table`` takes (int32 arrays, uint8 group ids)
    plus ``group_labels``."""
    teams = list(teams)
    T = len(teams)
    if T < 1:
        raise ValueError("the table has no teams")
    if T > SIM_MAX_TEAMS:
        raise ValueError(f"the table has {T} teams; at most {SIM_MAX_TEAMS} are supported")
    pw, pd = check_points(points)
    slot = {t: i for i, t in enumerate(teams)}
    pts, gf, ga = np.zeros(T, np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)
    if played is not None:
        ph, pa = _names(played["home_team"]), _names(played["away_team"])
        hg, ag = np.asarray(played["home_goals"]).astype(np.int64), np.asarray(played["away_goals"]).astype(np.int64)
        if not (len(ph) == len(pa) == len(hg) == len(ag)):
            raise ValueError("played: home_team, away_team, home_goals and away_goals differ in length")
        if (hg < 0).any() or (ag < 0).any():
            raise ValueError("played: goals must be non-negative")
        for h, a, x, y in zip(ph, pa, hg, ag):
            for t in (h, a):
                if t not in slot:
                    raise ValueError(f"played: team {t!r} is not in the table")
            if h == a:
                raise ValueError(f"played: team {h!r} plays itself")
            i, j = slot[h], slot[a]
            gf[i] += x
            ga[i] += y
            gf[j] += y
            ga[j] += x
            pts[i] += pw if x > y else pd if x == y else 0
            pts[j] += pw if y > x else pd if x == y else 0
    group, labels = None, None
    if groups is not None:
        lab = [groups[t] for t in teams] if isinstance(groups, dict) else list(groups)
        if len(lab) != T:
            raise ValueError(f"groups has {len(lab)} labels for {T} teams")
        labels = sorted(set(lab))
        ids = {g: k for k, g in enumerate(labels)}
        group = np.asarray([ids[g] for g in lab], np.uint8)
    return {"teams": teams, "start_points": pts.astype(np.int32), "start_goals_for": gf.astype(np.int32),
            "start_goals_against": ga.astype(np.int32), "group": group, "group_labels": labels,
            "points_win": pw, "points_draw": pd}


def fixture_slots(table: Dict[str, Any], home, away, known_teams=None) -> Tuple[np.ndarray, np.ndarray]:
    """Table slots (uint8) of the fixtures' teams.  Every team must be in the table and, when ``known_teams`` is given,
    known to the model; no team may play itself.  Also sets ``num_positions`` (the largest group) and
    ``num_points_bins`` (``points_win * max_t(remaining fixtures of t) + 1``) in ``table``."""
    home, away = _names(home), _names(away)
    if len(home) != len(away) or not home:
        raise ValueError("fixtures need home_team and away_team of the same, non-zero length")
    slot = {t: i for i, t in enumerate(table["teams"])}
    known = None if known_teams is None else set(np.asarray(known_teams).tolist())
    for h, a in zip(home, away):
        for t in (h, a):
            if known is not None and t not in known:
                raise ValueError(f"team {t!r} is not known to the model")
            if t not in slot:
                raise ValueError(f"team {t!r} plays a fixture but is not in the table")
        if h == a:
            raise ValueError(f"team {h!r} plays itself")
    hs = np.asarray([slot[t] for t in home], np.uint8)
    as_ = np.asarray([slot[t] for t in away], np.uint8)
    T = len(table["teams"])
    rem = np.bincount(hs, minlength=T) + np.bincount(as_, minlength=T)
    table["num_points_bins"] = int(table["points_win"] * rem.max() + 1)
    table["num_positions"] = T if table["group"] is None else int(np.bincount(table["group"]).max())
    return hs, as_


def probabilities(table: Dict[str, Any], position_counts: np.ndarray, points_counts: np.ndarray,
                  num_simulations: int) -> Dict[str, np.ndarray]:
    """Counts -> ``position_proba [T, P]``, ``points_proba [T, B]`` (points gained in the remaining fixtures) and
    ``expected_points = start_points + sum_b b points_proba[:, b]``."""
    n = float(num_simulations)
    pos = np.asarray(position_counts, np.float64) / n
    pts = np.asarray(points_counts, np.float64) / n
    start = np.asarray(table["start_points"], np.int64)
    return {"position_proba": pos, "points_proba": pts,
            "expected_points": start + pts @ np.arange(pts.shape[1], dtype=np.float64)}
