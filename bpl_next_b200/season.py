"""Host arithmetic of season and group-stage simulation: the table, slots and groups in, probabilities out.

The simulation itself is the CUDA kernel behind ``problem.simulate_table`` (``csrc/simulate.cu``); this module builds its
inputs from team names and played results and turns its integer counts into probabilities.  Definition, in short (the
full text is in ``include/bplx.h``): every simulated season takes ONE posterior draw and plays every remaining fixture
with that draw's rates, so a team that is stronger in a draw is stronger in all of its matches of that season.  Teams
are ranked within their group by points, then by the table's ranking rule (``TIEBREAKS``): ``"goal_difference"`` (the
default: goal difference, goals for, then a random tie-break key) or ``"head_to_head"`` (the matches among the teams
level on points first, reapplied to those still level; then goal difference, goals for and the key).  Fair-play rules
are not modelled: ties left at the end are decided by lot.  ``build_bracket`` and
``bracket_probabilities`` do the same for a knockout bracket played after the group stage (``problem.simulate_tournament``).
"""
from __future__ import annotations

import itertools
from typing import Any, Dict, Optional, Sequence, Tuple

import numpy as np

from ._abi import (ENTRANT_BEST, ENTRANT_GROUP_POS, ENTRANT_LOSER, ENTRANT_SLOT, ENTRANT_WINNER, KO_MAX_ALLOC_GROUPS,
                   KO_MAX_BEST, KO_MAX_ROUNDS, KO_MAX_TIES, RANK_GOAL_DIFF, RANK_HEAD_TO_HEAD, SIM_MAX_TEAMS,
                   TIE_ONE_MATCH, TIE_ONE_MATCH_ET, TIE_TWO_LEGS)

TIE_FORMATS = {"one_match": TIE_ONE_MATCH, "extra_time": TIE_ONE_MATCH_ET, "two_legs": TIE_TWO_LEGS}
TIEBREAKS = {"goal_difference": RANK_GOAL_DIFF, "head_to_head": RANK_HEAD_TO_HEAD}


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


def build_table(teams: Sequence, played: Optional[Dict[str, Any]] = None, groups=None, points=(3, 1),
                tiebreak: str = "goal_difference") -> Dict[str, Any]:
    """Starting table of ``teams`` from ``played`` results (reference ``training_data`` keys: ``home_team``,
    ``away_team``, ``home_goals``, ``away_goals``): points (``points = (win, draw)``), goals for and against.  ``groups``
    is a mapping team -> label or a sequence of labels aligned with ``teams`` (None: one table); labels become ids
    0 .. K-1 in sorted order.  ``tiebreak``: how teams level on points are ranked, ``"goal_difference"`` or
    ``"head_to_head"`` (``include/bplx.h``, BPLX_RANK_*).  Returns the host table ``problem.simulate_table`` takes
    (int32 arrays, uint8 group ids) plus ``group_labels`` and ``tiebreak``; under ``"head_to_head"`` also
    ``played_h2h`` (int32 ``[T, T, 2]``: points and goals of team u against team v in ``played``)."""
    if tiebreak not in TIEBREAKS:
        raise ValueError(f"unknown tiebreak {tiebreak!r} (one of {sorted(TIEBREAKS)})")
    teams = list(teams)
    T = len(teams)
    if T < 1:
        raise ValueError("the table has no teams")
    if T > SIM_MAX_TEAMS:
        raise ValueError(f"the table has {T} teams; at most {SIM_MAX_TEAMS} are supported")
    pw, pd = check_points(points)
    slot = {t: i for i, t in enumerate(teams)}
    pts, gf, ga = np.zeros(T, np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)
    h2h = np.zeros((T, T, 2), np.int64)
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
            pi, pj = (pw if x > y else pd if x == y else 0), (pw if y > x else pd if x == y else 0)
            pts[i] += pi
            pts[j] += pj
            h2h[i, j] += (pi, x)
            h2h[j, i] += (pj, y)
    group, labels = None, None
    if groups is not None:
        lab = [groups[t] for t in teams] if isinstance(groups, dict) else list(groups)
        if len(lab) != T:
            raise ValueError(f"groups has {len(lab)} labels for {T} teams")
        labels = sorted(set(lab))
        ids = {g: k for k, g in enumerate(labels)}
        group = np.asarray([ids[g] for g in lab], np.uint8)
    out = {"teams": teams, "start_points": pts.astype(np.int32), "start_goals_for": gf.astype(np.int32),
           "start_goals_against": ga.astype(np.int32), "group": group, "group_labels": labels,
           "points_win": pw, "points_draw": pd, "tiebreak": tiebreak}
    if tiebreak == "head_to_head":
        out["played_h2h"] = h2h.astype(np.int32)
    return out


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
    _size_histograms(table, hs, as_)
    return hs, as_


def _size_histograms(table: Dict[str, Any], home_slot=(), away_slot=()) -> None:
    """Sets ``num_positions`` (the largest group) and ``num_points_bins`` (``points_win * max_t(remaining fixtures of
    t) + 1``: 1 when there are no fixtures) in ``table`` for the fixtures between these slots."""
    T = len(table["teams"])
    rem = np.bincount(np.concatenate([home_slot, away_slot]).astype(np.int64), minlength=T)
    table["num_points_bins"] = int(table["points_win"] * rem.max() + 1)
    table["num_positions"] = T if table["group"] is None else int(np.bincount(table["group"]).max())


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


# ---- tournament: a knockout bracket after the group stage ---------------------------------------------------------
def _group_sizes(table: Dict[str, Any]) -> Tuple[list, np.ndarray]:
    """Group labels (``[None]`` for a table without groups) and the size of each group."""
    T = len(table["teams"])
    if table.get("group") is None:
        return [None], np.asarray([T])
    return list(table["group_labels"]), np.bincount(table["group"], minlength=len(table["group_labels"]))


def build_bracket(table: Dict[str, Any], ties: Sequence[Dict[str, Any]], best: Optional[Dict[str, Any]] = None
                  ) -> Dict[str, Any]:
    """The knockout bracket ``problem.simulate_tournament`` takes, from ties in play order.

    Each tie is ``{"id", "round", "home", "away", "neutral_venue", "format"}`` (``neutral_venue`` optional, default 0;
    ``format`` optional: ``"one_match"`` (default: one match, a draw decided by the per-draw win masses),
    ``"extra_time"`` (one match, then extra time and penalties) or ``"two_legs"`` (``home`` hosts leg 1, ``away`` leg
    2; level on aggregate: extra time in leg 2, then penalties; not at a neutral venue)); an entrant
    is ``("group", label, position)`` (0-based position in the group; label None for a table without groups),
    ``("best", j)`` (the j-th best-placed qualifier), ``("winner", id)`` / ``("loser", id)`` of an earlier tie, or
    ``("team", name)`` (a table team already through).  Round labels are ordered by first appearance; the last tie is
    the final and must be alone in its round.  ``best``: ``{"position": p, "count": c, "allocation": None or
    {frozenset(group labels): [group label of BEST j for j < c]}}`` -- the best c of the teams placed p in their
    groups qualify, ranked across groups by points, goal difference, goals for, then lot; with an allocation every
    c-subset of the groups must have a row, and each row is a permutation of its subset.  ``slot_team`` / ``slot_conf``
    are left to the caller (they need the model's team and confederation indices).  ``tie_format`` holds the
    ``_abi.TIE_*`` byte of every tie."""
    teams = list(table["teams"])
    slot = {t: i for i, t in enumerate(teams)}
    labels, sizes = _group_sizes(table)
    gid = {g: k for k, g in enumerate(labels)}
    ties = list(ties)
    K = len(ties)
    if not 1 <= K <= KO_MAX_TIES:
        raise ValueError(f"a bracket has 1 to {KO_MAX_TIES} ties, got {K}")
    bp, bc, alloc = 0, 0, None
    if best is not None:
        bp, bc, alloc = int(best["position"]), int(best["count"]), best.get("allocation")
        if not 1 <= bc <= min(KO_MAX_BEST, len(labels)):
            raise ValueError(f"best count must be in [1, {min(KO_MAX_BEST, len(labels))}], got {bc}")
        if not 0 <= bp < int(sizes.max()):
            raise ValueError(f"best position {bp} is outside every group")
    index, rounds, used = {}, [], set()
    kind = np.zeros((K, 2), np.uint8)
    arg0 = np.zeros((K, 2), np.uint8)
    arg1 = np.zeros((K, 2), np.uint8)
    rnd = np.zeros(K, np.uint8)
    nv = np.zeros(K, np.uint8)
    fmt = np.zeros(K, np.uint8)
    for k, tie in enumerate(ties):
        tid = tie["id"]
        if tid in index:
            raise ValueError(f"tie id {tid!r} is used twice")
        if tie["round"] not in rounds:
            rounds.append(tie["round"])
        rnd[k] = rounds.index(tie["round"])
        nv[k] = 1 if tie.get("neutral_venue", 0) else 0
        f = tie.get("format", "one_match")
        if f not in TIE_FORMATS:
            raise ValueError(f"tie {tid!r}: unknown format {f!r} (one of {sorted(TIE_FORMATS)})")
        fmt[k] = TIE_FORMATS[f]
        if fmt[k] == TIE_TWO_LEGS and nv[k]:
            raise ValueError(f"tie {tid!r}: a two-legged tie cannot be at a neutral venue")
        for side, key in enumerate(("home", "away")):
            e = tuple(tie[key])
            src = e
            if e[0] == "group":
                _, g, p = e
                if g not in gid:
                    raise ValueError(f"tie {tid!r}: unknown group {g!r}")
                if not 0 <= int(p) < sizes[gid[g]]:
                    raise ValueError(f"tie {tid!r}: group {g!r} has no position {p}")
                kind[k, side], arg0[k, side], arg1[k, side] = ENTRANT_GROUP_POS, gid[g], int(p)
                src = ("group", g, int(p))
            elif e[0] == "best":
                j = int(e[1])
                if not 0 <= j < bc:
                    raise ValueError(f"tie {tid!r}: best {j} is not one of the {bc} best-placed qualifiers")
                kind[k, side], arg0[k, side] = ENTRANT_BEST, j
                src = ("best", j)
            elif e[0] in ("winner", "loser"):
                ref = e[1]
                if ref not in index:
                    if any(t["id"] == ref for t in ties[k:]):
                        raise ValueError(f"tie {tid!r} refers to tie {ref!r}, which is not played before it")
                    raise ValueError(f"tie {tid!r} refers to an unknown tie id {ref!r}")
                kind[k, side] = ENTRANT_WINNER if e[0] == "winner" else ENTRANT_LOSER
                arg0[k, side] = index[ref]
            elif e[0] == "team":
                if e[1] not in slot:
                    raise ValueError(f"tie {tid!r}: team {e[1]!r} is not in the table")
                kind[k, side], arg0[k, side] = ENTRANT_SLOT, slot[e[1]]
            else:
                raise ValueError(f"tie {tid!r}: unknown entrant {e!r}")
            if src in used:
                raise ValueError(f"tie {tid!r}: entrant {src!r} is used twice")
            used.add(src)
        index[tid] = k
    if len(rounds) > KO_MAX_ROUNDS:
        raise ValueError(f"a bracket has at most {KO_MAX_ROUNDS} rounds, got {len(rounds)}")
    if (rnd == rnd[-1]).sum() != 1:
        raise ValueError(f"the last tie is the final and must be alone in its round {rounds[rnd[-1]]!r}")
    best_alloc = None
    if alloc is not None:
        ng = len(labels)
        if ng > KO_MAX_ALLOC_GROUPS:
            raise ValueError(f"an allocation table supports at most {KO_MAX_ALLOC_GROUPS} groups, got {ng}")
        best_alloc = np.full((1 << ng, bc), 0xFF, np.uint8)
        rows = {frozenset(k): list(v) for k, v in alloc.items()}
        for sub in itertools.combinations(range(ng), bc):
            key = frozenset(labels[g] for g in sub)
            if key not in rows:
                raise ValueError(f"the allocation misses the qualifying groups {sorted(key, key=str)}")
            row = rows[key]
            if len(row) != bc or set(row) != key:
                raise ValueError(f"allocation row {sorted(key, key=str)}: {row!r} is not a permutation of its groups")
            best_alloc[sum(1 << g for g in sub)] = [gid[g] for g in row]
        extra = [k for k in rows if len(k) != bc or not k <= set(labels)]
        if extra:
            raise ValueError(f"the allocation has a row for {sorted(extra[0], key=str)}, not {bc} of the table's groups")
    return {"ids": [t["id"] for t in ties], "rounds": rounds, "num_rounds": len(rounds), "kind": kind, "arg0": arg0,
            "arg1": arg1, "round": rnd, "neutral_venue": nv, "num_groups": len(labels), "best_position": bp,
            "best_count": bc, "best_alloc": best_alloc, "tie_format": fmt}


def bracket_probabilities(bracket: Dict[str, Any], reach_counts: np.ndarray, win_counts: np.ndarray,
                          num_simulations: int, decided_counts: Optional[np.ndarray] = None) -> Dict[str, Any]:
    """Counts -> ``reach_proba`` / ``win_proba [T, rounds]`` (a team reaches / wins a tie of the round),
    ``champion_proba [T]`` (it wins the last tie), ``tie_ids`` and, from ``decided_counts``, ``decided_proba [K, 3]``
    (tie k settled in normal time or on aggregate / in extra time / by the decider: penalties, or the per-draw lot of a
    ``one_match`` tie)."""
    n = float(num_simulations)
    reach = np.asarray(reach_counts, np.float64) / n
    win = np.asarray(win_counts, np.float64) / n
    return {"rounds": list(bracket["rounds"]), "reach_proba": reach, "win_proba": win,
            "champion_proba": win[:, int(bracket["round"][-1])].copy(), "tie_ids": list(bracket["ids"]),
            "decided_proba": None if decided_counts is None else np.asarray(decided_counts, np.float64) / n}
