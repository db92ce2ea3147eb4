"""Restatement of the tournament simulation (``csrc/simulate.cu``, ``simulate_kernel<true>``) in float64 numpy.

TEST INFRASTRUCTURE ONLY.  It builds on the season / group-stage restatement of ``oracle/simulate.py`` (same Philox
words, same score walks, same ranking) and adds the knockout bracket.

Definition (the same text as ``include/bplx.h``): the group stage of ``oracle/simulate.py``, then K ties in play order.
An entrant is a fixed slot, the slot ranked p in group g, the j-th best-placed qualifier, or the winner / loser of an
earlier tie.  Best-placed qualifiers: the slots at ``best_position`` of every group, ranked across groups by points,
goal difference, goals for, the slot tie-break key (word ``2F + t``), then the lower slot; the first ``best_count``
qualify; with an allocation table ``[2^num_groups, best_count]`` BEST j is the position-``best_position`` slot of group
``alloc[mask, j]`` (mask = the bit set of the qualifying groups).  A tie is played like a group fixture from the draw's
own grid (words ``2F + T_tab + 3k`` and ``+ 1``); a drawn tie goes to the home entrant iff ``u_d (hw + aw) <= hw``
(word ``+ 2``), ``hw = sum_{i > j} w(i, j)``, ``aw = sum_{i < j} w(i, j)``.  Extra time, penalties, fair play and
head-to-head are not modelled.  A tie with a non-finite rate or normaliser, ``hw + aw`` not positive on a drawn tie, a
group position beyond its group, fewer than ``best_count`` candidates or an allocation entry of 0xFF makes the
simulation invalid.

``resolve_bracket`` is the bracket in pure integer logic from given scores and decider outcomes; ``simulate_tournament``
replays the kernel on the same Philox words and returns a per-tie margin for the score walks and for the decider,
``|u_d (hw + aw) - hw| / (hw + aw)``: the float32 kernel may differ from it only where a margin is at rounding level.
"""
from __future__ import annotations

import numpy as np

from oracle import philox
from oracle import predict as op
from oracle.simulate import _pmf_unnormalised, rank, rank_scores, sample_scores, simulate, tables

SLOT, GROUP_POS, BEST, WINNER, LOSER = 0, 1, 2, 3, 4


def _group_layout(table, num_groups):
    g = np.zeros(len(table["start_points"]), np.int64) if table.get("group") is None else np.asarray(table["group"],
                                                                                                      np.int64)
    return g, np.bincount(g, minlength=num_groups)[:num_groups]


def qualifiers(table, bracket, pts, gd, gf, keys, pos):
    """Per simulation: ``qmap [n, groups, P]`` (slot ranked p in group g, -1 where the group has none) and the
    best-placed slots ``best [n, best_count]`` (-1 where the simulation is invalid), and a validity flag."""
    n, T = pos.shape
    ng = int(bracket["num_groups"])
    group, sizes = _group_layout(table, ng)
    P = int(pos.max(initial=0)) + 1 if pos.size else 1
    qmap = np.full((n, max(ng, 1), max(P, T)), -1, np.int64)
    for t in range(T):
        if group[t] < ng:
            qmap[np.arange(n), group[t], pos[:, t]] = t
    bc, bp = int(bracket["best_count"]), int(bracket["best_position"])
    best = np.full((n, max(bc, 1)), -1, np.int64)
    ok = np.ones(n, bool)
    if bc == 0:
        return qmap, best, ok
    alloc = bracket.get("best_alloc")
    cand_groups = [g for g in range(ng) if sizes[g] > bp]
    for i in range(n):
        cands = [(g, qmap[i, g, bp]) for g in cand_groups]
        order = sorted(cands, key=lambda c: (-pts[i, c[1]], -gd[i, c[1]], -gf[i, c[1]], -keys[i, c[1]], c[1]))[:bc]
        if len(order) < bc:
            ok[i] = False
            continue
        if alloc is None:
            best[i] = [c[1] for c in order]
            continue
        mask = sum(1 << g for g, _ in order)
        row = np.asarray(alloc)[mask]
        if any(r >= ng or not (mask >> int(r)) & 1 for r in row):
            ok[i] = False
            continue
        best[i] = qmap[i, row.astype(np.int64), bp]
    return qmap, best, ok


def _play_bracket(table, bracket, pts, gd, gf, keys, pos, valid, play_tie):
    """The bracket of every simulation; ``play_tie(k, home_slot [n], away_slot [n], live [n])`` returns
    ``(home_goals, away_goals, home_through, ok)`` ``[n]`` for tie k."""
    n, T = pos.shape
    K, nr = len(bracket["round"]), int(bracket["num_rounds"])
    _, sizes = _group_layout(table, int(bracket["num_groups"]))
    qmap, best, ok = qualifiers(table, bracket, pts, gd, gf, keys, np.where(valid[:, None], pos, 0))
    ok &= valid
    kind, a0, a1 = (np.asarray(bracket[k], np.int64) for k in ("kind", "arg0", "arg1"))
    ent = np.zeros((n, K, 2), np.int64)
    ksc = np.zeros((n, K, 2), np.int64)
    win = np.zeros((n, K), np.int64)
    lose = np.zeros((n, K), np.int64)
    rows = np.arange(n)
    for k in range(K):
        for side in range(2):
            kd, x, y = kind[k, side], a0[k, side], a1[k, side]
            if kd == SLOT:
                e = np.full(n, x)
            elif kd == GROUP_POS:
                inside = y < sizes[x]
                ok &= inside
                e = qmap[:, x, y] if inside else np.zeros(n, np.int64)
            elif kd == BEST:
                e = best[:, x]
            elif kd == WINNER:
                e = win[:, x]
            else:
                e = lose[:, x]
            ent[:, k, side] = np.where(ok, e, 0)
        hg, ag, through, tok = play_tie(k, ent[:, k, 0], ent[:, k, 1], ok.copy())
        ok &= tok
        ksc[:, k, 0], ksc[:, k, 1] = hg, ag
        w_home = np.where(hg == ag, through, hg > ag)
        win[:, k] = np.where(w_home, ent[:, k, 0], ent[:, k, 1])
        lose[:, k] = np.where(w_home, ent[:, k, 1], ent[:, k, 0])
    reach = np.zeros((T, nr), np.int64)
    wins = np.zeros((T, nr), np.int64)
    rnd = np.asarray(bracket["round"], np.int64)
    for k in range(K):
        np.add.at(reach, (win[ok, k], rnd[k]), 1)
        np.add.at(reach, (lose[ok, k], rnd[k]), 1)
        np.add.at(wins, (win[ok, k], rnd[k]), 1)
    bad = ~ok[:, None, None]
    return {"ko_entrants": np.where(bad, 255, ent), "ko_scores": np.where(bad, 255, ksc),
            "ko_winners": np.where(~ok[:, None], 255, win), "reach_counts": reach, "win_counts": wins, "valid": ok}


def resolve_bracket(table, home_slot, away_slot, bracket, home, away, keys, ko_home, ko_away, home_through,
                    valid=None):
    """The bracket in pure integer logic from given scores: group scores ``home`` / ``away [n, F]``, tie-break keys
    ``[n, T]``, tie scores ``ko_home`` / ``ko_away [n, K]`` and ``home_through [n, K]`` (whether the home entrant won
    the decider; read only for drawn ties).  Returns ``rank_scores``'s outputs restricted to the simulations the bracket
    leaves valid, ``ko_entrants [n, K, 2]``, ``ko_scores``, ``ko_winners [n, K]`` (255 for invalid simulations),
    ``reach_counts`` / ``win_counts [T, rounds]``, ``valid [n]`` and ``invalid``."""
    n = np.asarray(keys).shape[0]
    valid = np.ones(n, bool) if valid is None else np.asarray(valid, bool)
    home, away = np.asarray(home, np.int64), np.asarray(away, np.int64)
    hv, av = np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0)
    pts, gd, gf = tables(table, home_slot, away_slot, hv, av)
    keys = np.asarray(keys, np.int64)
    pos = rank(pts, gd, gf, keys, table.get("group"))
    kh, ka, th = (np.asarray(x).astype(np.int64) for x in (ko_home, ko_away, home_through))

    def play(k, hs, as_, live):
        return kh[:, k], ka[:, k], th[:, k].astype(bool), np.ones(n, bool)

    out = _play_bracket(table, bracket, pts, gd, gf, keys, pos, valid, play)
    r = rank_scores(table, home_slot, away_slot, home, away, keys, out["valid"])
    out.update(r, invalid=int((~out["valid"]).sum()))
    return out


def win_masses(lh, la, c, max_goals):
    """The draw's un-normalised ``hw = sum_{i > j} w(i, j)`` and ``aw = sum_{i < j} w(i, j)`` (tau clamped), ``[n]``."""
    G = int(max_goals)
    p, q = _pmf_unnormalised(lh, G), _pmf_unnormalised(la, G)
    with np.errstate(over="ignore", invalid="ignore"):
        w = p[:, :, None] * q[:, None, :]
        w[:, 0, 1] *= np.maximum(1.0 + c * lh, 0.0)
        w[:, 1, 0] *= np.maximum(1.0 + c * la, 0.0)
        low = np.tril(np.ones((G + 1, G + 1), bool), -1)  # i > j
        return (w * low).sum(axis=(1, 2)), (w * low.T).sum(axis=(1, 2))


def simulate_tournament(model, samples, fixtures, home_slot, away_slot, table, bracket, max_goals, sims_per_draw, seed,
                        first_draw=0):
    """The tournaments of draws ``samples`` replayed on the kernel's Philox words: ``simulate``'s outputs for the
    group stage plus ``_play_bracket``'s, ``ko_margin [N, K]`` (the score walks' margin of each tie) and
    ``decider_margin [N, K]`` (``|u_d (hw + aw) - hw| / (hw + aw)`` on drawn ties, inf elsewhere)."""
    F = 0 if fixtures is None or fixtures.get("home_team") is None else len(fixtures["home_team"])
    T = len(table["start_points"])
    K = len(bracket["round"])
    R = int(sims_per_draw)
    S = np.asarray(samples["attack"]).shape[0]
    N = S * R
    if F:
        g = simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, R, seed, first_draw)
    else:
        g = {"home": np.zeros((N, 0), np.int64), "away": np.zeros((N, 0), np.int64), "valid": np.ones(N, bool),
             "margin": np.zeros((N, 0))}
        hs0 = np.zeros(0, np.int64)
        home_slot = away_slot = hs0
    s_of = np.repeat(np.arange(S), R)
    n_glob = (first_draw + s_of) * R + np.tile(np.arange(R), S)
    words = philox.stream(int(seed), n_glob.astype(np.uint64), 0, 2 * F + T + 3 * K)
    keys = words[:, 2 * F:2 * F + T].astype(np.int64)
    u = philox.uniform(words[:, 2 * F + T:]).astype(np.float64)
    valid = g["valid"]
    hv, av = np.where(valid[:, None], g["home"], 0), np.where(valid[:, None], g["away"], 0)
    pts, gd, gf = tables(table, np.minimum(home_slot, T - 1), np.minimum(away_slot, T - 1), hv, av)
    pos = rank(pts, gd, gf, keys, table.get("group"))
    # the rates of every ordered pair of slots, at home and at a neutral venue: [S, T * T]
    st = np.asarray(bracket["slot_team"], np.int64)
    ht, at = np.repeat(st, T), np.tile(st, T)
    kw = {}
    if model == "neutral_wc":
        sc = np.asarray(bracket["slot_conf"], np.int64)
        kw = {"home_conf": np.repeat(sc, T), "away_conf": np.tile(sc, T)}
    rates = {}
    for nv in (0, 1):
        extra = dict(kw, neutral_venue=np.full(T * T, nv, np.uint8)) if model in ("neutral", "neutral_wc") else kw
        with np.errstate(over="ignore", invalid="ignore"):
            rates[nv] = op.expected_goals(model, samples, ht, at, **extra)
    cc = np.asarray(samples["corr_coef"], np.float64)[s_of]
    nvk = np.asarray(bracket.get("neutral_venue") if bracket.get("neutral_venue") is not None else np.zeros(K), np.int64)
    ko_margin = np.full((N, K), np.inf)
    dec_margin = np.full((N, K), np.inf)

    def play(k, hs, as_, live):
        lh, la = (r[s_of, hs * T + as_] for r in rates[int(nvk[k] and model in ("neutral", "neutral_wc"))])
        h, a, m, v = sample_scores(lh, la, cc, u[:, 3 * k], u[:, 3 * k + 1], max_goals)
        ko_margin[:, k] = np.where(live, m, np.inf)
        hw, aw = win_masses(lh, la, cc, max_goals)
        tot = hw + aw
        drawn = v & (h == a)
        v &= ~drawn | (tot > 0)
        with np.errstate(invalid="ignore", divide="ignore"):
            through = u[:, 3 * k + 2] * tot <= hw
            dec_margin[:, k] = np.where(live & drawn, np.abs(u[:, 3 * k + 2] * tot - hw) / tot, np.inf)
        return h, a, through, v

    out = _play_bracket(table, bracket, pts, gd, gf, keys, pos, valid, play)
    r = rank_scores(table, np.minimum(home_slot, T - 1), np.minimum(away_slot, T - 1), g["home"], g["away"], keys,
                    out["valid"])
    out.update(r, home=g["home"], away=g["away"], margin=g["margin"], keys=keys, ko_margin=ko_margin,
               decider_margin=dec_margin,
               invalid=int((~out["valid"]).sum()))
    return out
