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
``build_conditions`` and ``conditional_probabilities`` give match importance: finishing probabilities conditioned on the
outcome of key fixtures (``problem.simulate_table(conditions=...)``).
"""
from __future__ import annotations

import itertools
from typing import Any, Dict, Optional, Sequence, Tuple

import numpy as np

from ._abi import (ENTRANT_BEST, ENTRANT_GROUP_POS, ENTRANT_LOSER, ENTRANT_PAIRED, ENTRANT_SLOT, ENTRANT_WINNER,
                   KO_MAX_ALLOC_GROUPS, KO_MAX_BEST, KO_MAX_ROUNDS, KO_MAX_TIES, MAX_PAIRINGS, PAIRING_MAX_POOL,
                   PAIRING_MAX_POT, PAIRING_OPEN, PAIRING_SEEDED, PROTECT_ASSOCIATION, PROTECT_GROUP, RANK_GOAL_DIFF,
                   RANK_HEAD_TO_HEAD, SIM_MAX_EVENTS, SIM_MAX_KEY_FIXTURES, SIM_MAX_TEAMS, TIE_ONE_MATCH, TIE_ONE_MATCH_ET,
                   TIE_TWO_LEGS)

TIE_FORMATS = {"one_match": TIE_ONE_MATCH, "extra_time": TIE_ONE_MATCH_ET, "two_legs": TIE_TWO_LEGS}
TIEBREAKS = {"goal_difference": RANK_GOAL_DIFF, "head_to_head": RANK_HEAD_TO_HEAD}
PROTECTIONS = {"group": PROTECT_GROUP, "association": PROTECT_ASSOCIATION}


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


# ---- match importance: finishing probabilities conditioned on key fixtures' results ----------------------------------
def build_conditions(table: Dict[str, Any], num_fixtures: int, key_fixtures: Sequence[int],
                     events: Dict[Any, Tuple[Any, Any]]) -> Dict[str, Any]:
    """The conditions ``problem.simulate_table`` takes, from fixture indices and events on team names.

    Key fixture j has outcome o in {0 home win, 1 draw, 2 away win}, taken from its sampled score; event e = (team,
    positions) holds in a simulation iff the team's 0-based position within its group is one of ``positions`` (an int or
    an iterable).  ``key_fixtures``: distinct indices into the ``num_fixtures`` fixtures, in any order and any number;
    ``events``: label -> (team, positions), 1 to 64 of them.  Returns ``key_fixtures`` and ``events`` (the labels) in
    the caller's order, ``event_slot`` (uint8 ``[E]``), ``event_positions`` (uint64 ``[E]``, bit p = position p) and
    ``groups``: the key fixtures sorted and cut into runs of at most 64, each ``{"key_fixture": int32 [Kc], "rows":
    int64 [Kc]}`` with ``rows`` the index in ``key_fixtures`` of each key.  Each run is one simulation."""
    keys = [int(k) for k in key_fixtures]
    if not keys:
        raise ValueError("key_fixtures is empty")
    for k in keys:
        if not 0 <= k < num_fixtures:
            raise ValueError(f"key fixture {k} is not one of the {num_fixtures} fixtures")
    if len(set(keys)) != len(keys):
        raise ValueError("key_fixtures lists a fixture more than once")
    events = dict(events)
    if not 1 <= len(events) <= SIM_MAX_EVENTS:
        raise ValueError(f"between 1 and {SIM_MAX_EVENTS} events are supported, got {len(events)}")
    slot = {t: i for i, t in enumerate(table["teams"])}
    labels, sizes = _group_sizes(table)
    group = np.zeros(len(slot), np.int64) if table.get("group") is None else np.asarray(table["group"], np.int64)
    eslot = np.zeros(len(events), np.uint8)
    emask = np.zeros(len(events), np.uint64)
    for e, (label, ev) in enumerate(events.items()):
        try:
            team, positions = ev
        except (TypeError, ValueError):
            raise ValueError(f"event {label!r}: expected (team, positions), got {ev!r}") from None
        if team not in slot:
            raise ValueError(f"event {label!r}: team {team!r} is not in the table")
        size = int(sizes[group[slot[team]]])
        pos = [positions] if isinstance(positions, (int, np.integer)) else list(positions)
        if not pos:
            raise ValueError(f"event {label!r}: no positions")
        m = 0
        for p in pos:
            if not isinstance(p, (int, np.integer)) or isinstance(p, bool) or not 0 <= p < size:
                raise ValueError(f"event {label!r}: position {p!r} is not a position of a group of {size}")
            m |= 1 << int(p)
        eslot[e], emask[e] = slot[team], m
    order = np.argsort(keys, kind="stable")
    groups = [{"key_fixture": np.asarray([keys[i] for i in order[lo:lo + SIM_MAX_KEY_FIXTURES]], np.int32),
               "rows": order[lo:lo + SIM_MAX_KEY_FIXTURES].astype(np.int64)}
              for lo in range(0, len(keys), SIM_MAX_KEY_FIXTURES)]
    return {"key_fixtures": keys, "events": list(events), "event_slot": eslot, "event_positions": emask,
            "groups": groups}


def conditional_probabilities(conditions: Dict[str, Any], outcome_counts: np.ndarray, conditional_counts: np.ndarray,
                              num_simulations: int) -> Dict[str, Any]:
    """Counts -> ``outcome_proba [Kc, 3]`` (key fixture j ends in a home win / draw / away win), ``event_proba [E]``,
    ``conditional_proba [Kc, 3, E]`` (P(event e | key fixture j ended in o); NaN where o never occurred) and
    ``importance [Kc, E]`` (the largest minus the smallest ``conditional_proba`` over the outcomes that occurred; 0 if
    fewer than two occurred), with ``key_fixtures``, ``events`` and the integer counts.  Rows follow
    ``conditions["key_fixtures"]``."""
    oc = np.asarray(outcome_counts, np.int64)
    cc = np.asarray(conditional_counts, np.int64)
    n = float(num_simulations)
    seen = oc > 0
    with np.errstate(invalid="ignore", divide="ignore"):
        cond = np.where(seen[:, :, None], cc / oc[:, :, None].astype(np.float64), np.nan)
    hi = np.where(seen[:, :, None], cond, -np.inf).max(axis=1)
    lo = np.where(seen[:, :, None], cond, np.inf).min(axis=1)
    importance = np.where((seen.sum(axis=1) >= 2)[:, None], hi - lo, 0.0)
    return {"key_fixtures": list(conditions["key_fixtures"]), "events": list(conditions["events"]),
            "outcome_proba": oc / n, "event_proba": cc[0].sum(axis=0) / n, "conditional_proba": cond,
            "importance": importance, "outcome_counts": oc, "conditional_counts": cc}


# ---- tournament: a knockout bracket after the group stage ---------------------------------------------------------
def _group_sizes(table: Dict[str, Any]) -> Tuple[list, np.ndarray]:
    """Group labels (``[None]`` for a table without groups) and the size of each group."""
    T = len(table["teams"])
    if table.get("group") is None:
        return [None], np.asarray([T])
    return list(table["group_labels"]), np.bincount(table["group"], minlength=len(table["group_labels"]))


def build_bracket(table: Dict[str, Any], ties: Sequence[Dict[str, Any]], best: Optional[Dict[str, Any]] = None,
                  pairings: Optional[Sequence[Dict[str, Any]]] = None, association=None) -> Dict[str, Any]:
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
    ``_abi.TIE_*`` byte of every tie.

    ``pairings``: draws by lot that pair a pool of entrants when the first tie taking one of their pairs is reached
    (``include/bplx.h``, bplx_pairings), each ``{"id", "pool": [entrants], "pots": None or [0 / 1 per entrant],
    "protect": a set of "group" / "association", "seeded_home": bool}``.  ``pots`` None is an open draw (at most 64
    entrants, an even number, no protection): the pool is shuffled and the first team drawn of each pair is at home.
    With pots, pot 0 is seeded and pot 1 unseeded, at most 16 each and equal in size: UEFA's sequential procedure
    draws an unseeded team, then one of the seeded teams it may meet for which the rest can still be paired; the
    unseeded team is at home unless ``seeded_home``.  ``protect`` forbids pairs of the same group or of the same
    ``association`` (a mapping team -> label, or labels aligned with the table's teams; a team without one never
    clashes).  A tie takes pair i of a pairing with ``"pair": (pairing id, i)`` instead of ``home`` / ``away``; every
    pair feeds exactly one tie, and a pool's winners / losers must come from ties played before the first such tie."""
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
    def entrant(e, where):
        """(kind, arg0, arg1, source key) of entrant ``e``."""
        e = tuple(e)
        if e[0] == "group":
            _, g, p = e
            if g not in gid:
                raise ValueError(f"{where}: unknown group {g!r}")
            if not 0 <= int(p) < sizes[gid[g]]:
                raise ValueError(f"{where}: group {g!r} has no position {p}")
            return ENTRANT_GROUP_POS, gid[g], int(p), ("group", g, int(p))
        if e[0] == "best":
            j = int(e[1])
            if not 0 <= j < bc:
                raise ValueError(f"{where}: best {j} is not one of the {bc} best-placed qualifiers")
            return ENTRANT_BEST, j, 0, ("best", j)
        if e[0] in ("winner", "loser"):
            ref = e[1]
            if ref not in index:
                if any(t["id"] == ref for t in ties):
                    raise ValueError(f"{where} refers to tie {ref!r}, which is not played before it")
                raise ValueError(f"{where} refers to an unknown tie id {ref!r}")
            return ENTRANT_WINNER if e[0] == "winner" else ENTRANT_LOSER, index[ref], 0, e
        if e[0] == "team":
            if e[1] not in slot:
                raise ValueError(f"{where}: team {e[1]!r} is not in the table")
            return ENTRANT_SLOT, slot[e[1]], 0, e
        raise ValueError(f"{where}: unknown entrant {e!r}")

    def take(src, where):
        if src in used:
            raise ValueError(f"{where}: entrant {src!r} is used twice")
        used.add(src)

    pairings = None if pairings is None else list(pairings)
    P = 0 if pairings is None else len(pairings)
    if P > MAX_PAIRINGS:
        raise ValueError(f"a bracket has at most {MAX_PAIRINGS} pairings, got {P}")
    pid = {}
    for d, pg in enumerate(pairings or ()):
        if pg["id"] in pid:
            raise ValueError(f"pairing id {pg['id']!r} is used twice")
        pid[pg["id"]] = d
    pmode, pprot, phost, psize = (np.zeros(P, np.uint8) for _ in range(4))
    pkind, parg0, parg1, ppot = (np.zeros((P, PAIRING_MAX_POOL), np.uint8) for _ in range(4))
    made, taken = set(), [set() for _ in range(P)]

    def make_pairing(d):
        """Pairing d's pool, read when its first tie is reached (so its winners / losers are of earlier ties)."""
        pg = pairings[d]
        where = f"pairing {pg['id']!r}"
        pool, pots = list(pg["pool"]), pg.get("pots")
        n = len(pool)
        prot = 0
        for name in pg.get("protect") or ():
            if name not in PROTECTIONS:
                raise ValueError(f"{where}: unknown protection {name!r} (one of {sorted(PROTECTIONS)})")
            prot |= PROTECTIONS[name]
        if pots is None:
            if prot:
                raise ValueError(f"{where}: protections need a seeded draw (pots)")
            if not (2 <= n <= PAIRING_MAX_POOL and n % 2 == 0):
                raise ValueError(f"{where}: an open draw needs an even pool of 2 to {PAIRING_MAX_POOL}, got {n}")
        else:
            pots = [int(x) for x in pots]
            if len(pots) != n or any(x not in (0, 1) for x in pots):
                raise ValueError(f"{where}: pots must give 0 or 1 for every pool entrant")
            m = pots.count(0)
            if 2 * m != n or not 1 <= m <= PAIRING_MAX_POT:
                raise ValueError(f"{where}: the pots must be equal in size, 1 to {PAIRING_MAX_POT} each "
                                 f"(got {m} and {n - m})")
            if prot & PROTECT_GROUP and table.get("group") is None:
                raise ValueError(f"{where}: group protection needs a table with groups")
            if prot & PROTECT_ASSOCIATION and association is None:
                raise ValueError(f"{where}: association protection needs association")
        for j, e in enumerate(pool):
            kd, a0, a1, src = entrant(e, where)
            take(src, where)
            pkind[d, j], parg0[d, j], parg1[d, j] = kd, a0, a1
            ppot[d, j] = 0 if pots is None else pots[j]
        pmode[d] = PAIRING_OPEN if pots is None else PAIRING_SEEDED
        pprot[d], psize[d] = prot, n
        phost[d] = 0 if pots is None or pg.get("seeded_home", False) else 1
        made.add(d)

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
        if "pair" in tie:
            if "home" in tie or "away" in tie:
                raise ValueError(f"tie {tid!r}: a tie takes a pair or a home and an away entrant, not both")
            ref, i = tie["pair"]
            if ref not in pid:
                raise ValueError(f"tie {tid!r}: unknown pairing {ref!r}")
            d, i = pid[ref], int(i)
            if d not in made:
                make_pairing(d)
            if not 0 <= i < psize[d] // 2:
                raise ValueError(f"tie {tid!r}: pairing {ref!r} has no pair {i}")
            if i in taken[d]:
                raise ValueError(f"tie {tid!r}: pair {i} of pairing {ref!r} is taken twice")
            taken[d].add(i)
            kind[k] = ENTRANT_PAIRED
            arg0[k], arg1[k] = d, (2 * i, 2 * i + 1)
        else:
            for side, key in enumerate(("home", "away")):
                kind[k, side], arg0[k, side], arg1[k, side], src = entrant(tie[key], f"tie {tid!r}")
                take(src, f"tie {tid!r}")
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
    out = {"ids": [t["id"] for t in ties], "rounds": rounds, "num_rounds": len(rounds), "kind": kind, "arg0": arg0,
           "arg1": arg1, "round": rnd, "neutral_venue": nv, "num_groups": len(labels), "best_position": bp,
           "best_count": bc, "best_alloc": best_alloc, "tie_format": fmt}
    if pairings is not None:
        for d, pg in enumerate(pairings):
            if len(taken[d]) != psize[d] // 2:
                raise ValueError(f"pairing {pg['id']!r}: {psize[d] // 2 - len(taken[d])} of its pairs feed no tie")
        slot_assoc = None
        if association is not None:
            lab = [association.get(t) for t in teams] if isinstance(association, dict) else list(association)
            if len(lab) != len(teams):
                raise ValueError(f"association has {len(lab)} labels for {len(teams)} teams")
            ids = {a: i for i, a in enumerate(sorted({a for a in lab if a is not None}, key=str))}
            if len(ids) > 255:
                raise ValueError("at most 255 associations are supported")
            slot_assoc = np.asarray([0xFF if a is None else ids[a] for a in lab], np.uint8)
        out.update(pairing_ids=list(pid), pairing_mode=pmode, pairing_protect=pprot, pairing_host_pot=phost,
                   pool_size=psize, pool_kind=pkind, pool_arg0=parg0, pool_arg1=parg1, pool_pot=ppot,
                   slot_assoc=slot_assoc)
    return out


def bracket_probabilities(bracket: Dict[str, Any], reach_counts: np.ndarray, win_counts: np.ndarray,
                          num_simulations: int, decided_counts: Optional[np.ndarray] = None,
                          pairing_counts: Optional[np.ndarray] = None) -> Dict[str, Any]:
    """Counts -> ``reach_proba`` / ``win_proba [T, rounds]`` (a team reaches / wins a tie of the round),
    ``champion_proba [T]`` (it wins the last tie), ``tie_ids`` and, from ``decided_counts``, ``decided_proba [K, 3]``
    (tie k settled in normal time or on aggregate / in extra time / by the decider: penalties, or the per-draw lot of a
    ``one_match`` tie); from ``pairing_counts``, ``pairing_ids`` and ``pairing_proba [P, T, T]`` (pairing d drew team
    u at home against team v)."""
    n = float(num_simulations)
    reach = np.asarray(reach_counts, np.float64) / n
    win = np.asarray(win_counts, np.float64) / n
    out = {"rounds": list(bracket["rounds"]), "reach_proba": reach, "win_proba": win,
           "champion_proba": win[:, int(bracket["round"][-1])].copy(), "tie_ids": list(bracket["ids"]),
           "decided_proba": None if decided_counts is None else np.asarray(decided_counts, np.float64) / n}
    if pairing_counts is not None:
        out.update(pairing_ids=list(bracket["pairing_ids"]),
                   pairing_proba=np.asarray(pairing_counts, np.float64) / n)
    return out
