"""Restatement of the tournament simulation (``csrc/simulate.cu``, ``simulate_kernel<true>``) in float64 numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  It builds on the season / group-stage restatement of
``oracle/simulate.py`` (same Philox words, same score walks, same ranking) and adds the knockout bracket.

Definition (the same text as ``include/bplx.h``): the group stage of ``oracle/simulate.py``, then K ties in play order.
An entrant is a fixed slot, the slot ranked p in group g, the j-th best-placed qualifier, or the winner / loser of an
earlier tie.  Best-placed qualifiers: the slots at ``best_position`` of every group, ranked across groups by points,
goal difference, goals for, the slot tie-break key (word ``2F + t``), then the lower slot; the first ``best_count``
qualify; with an allocation table ``[2^num_groups, best_count]`` BEST j is the position-``best_position`` slot of group
``alloc[mask, j]`` (mask = the bit set of the qualifying groups).  Each tie has a format byte
(``bracket["tie_format"]``, all 0 when absent):

  0 BPLX_TIE_ONE_MATCH     one match; a draw is decided by ``u_d (hw + aw) <= hw``
  1 BPLX_TIE_ONE_MATCH_ET  one match; drawn: extra time; still level: penalties
  2 BPLX_TIE_TWO_LEGS      two legs; level on aggregate: extra time in leg 2; still level: penalties

A match is played like a group fixture from the draw's own grid.  ``hw = sum_{i > j} w(i, j)``,
``aw = sum_{i < j} w(i, j)``.  The home entrant A hosts leg 1, the away entrant B leg 2 with the venues swapped
(neutral_venue 0 in both legs; for NeutralWC the confederations swap sides).  Aggregate ``A = h1 + a2``,
``B = a1 + h2``; the higher goes through, no away-goals rule.  Extra time is played at the venue of the last match
(format 1: with the tie's neutral flag) on the draw's rates times ``EXTRA_TIME_FRACTION = 1/3``, without the tau
correction (independent Poissons truncated at G).  Penalties: A goes through iff ``u_d <= 1/2``.  Fair play and
head-to-head are not modelled.  Tie k reads words ``2F + T_tab + 3k`` and ``+ 1`` (its first or only match) and ``+ 2``
(``u_d``); with ``E = 4 ceil((2F + T_tab + 3K) / 4)`` it owns words ``E + 4k .. E + 4k + 3``: leg 2 ``(u_h, u_a)``,
then extra time ``(u_h, u_a)``.  A non-finite rate or normaliser in any match of a tie, ``hw + aw`` not positive on a
drawn format-0 tie, a group position beyond its group, fewer than ``best_count`` candidates or an allocation entry of
0xFF makes the simulation invalid.

``resolve_bracket`` is the bracket in pure integer logic from given scores and decider outcomes; ``simulate_tournament``
replays the kernel on the same Philox words and returns a per-tie margin for the score walks of every match and for
the decider (``|u_d (hw + aw) - hw| / (hw + aw)``, or ``|u_d - 1/2|`` for penalties): the float32 kernel may differ
from it only where a margin is at rounding level.  ``tie_closed_form`` gives, per draw, P(A through), P(extra time) and
P(penalties) of one tie between two fixed teams by convolving goal-difference distributions.
"""
from __future__ import annotations

import numpy as np

from oracle import philox
from oracle import predict as op
from oracle.simulate import _pmf_unnormalised, histograms, philox_words, play_fixtures, rank, sample_scores, tables

SLOT, GROUP_POS, BEST, WINNER, LOSER = 0, 1, 2, 3, 4
ONE_MATCH, ONE_MATCH_ET, TWO_LEGS = 0, 1, 2
EXTRA_TIME_FRACTION = 1.0 / 3.0
NOT_PLAYED = 254


def _group_layout(table, num_groups):
    g = np.zeros(len(table["start_points"]), np.int64) if table.get("group") is None else np.asarray(table["group"],
                                                                                                      np.int64)
    return g, np.bincount(g, minlength=num_groups)[:num_groups]


def _formats(bracket):
    K = len(bracket["round"])
    f = bracket.get("tie_format")
    return np.zeros(K, np.int64) if f is None else np.asarray(f, np.int64)


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


def settle(fmt, h1, a1, extra, decider):
    """How a tie of format ``fmt`` ends, from the first (or only) match ``h1``, ``a1`` (home entrant A, away entrant
    B), ``extra [n, 4]`` (leg-2 goals of A and B, extra-time goals of A and B) and the decider outcome ``decider [n]``
    (A through on u_d: the lot of format 0, else penalties).  Returns ``(A through [n], how [n])``, how = 0 (normal
    time or aggregate), 1 (extra time), 2 (the decider)."""
    extra = np.asarray(extra, np.int64)
    ta, tb = np.asarray(h1, np.int64), np.asarray(a1, np.int64)
    if fmt == TWO_LEGS:
        ta, tb = ta + extra[:, 0], tb + extra[:, 1]
    level = ta == tb
    if fmt == ONE_MATCH:
        return np.where(level, decider, ta > tb), np.where(level, 2, 0)
    ta, tb = ta + np.where(level, extra[:, 2], 0), tb + np.where(level, extra[:, 3], 0)
    still = level & (ta == tb)
    return np.where(still, decider, ta > tb), np.where(still, 2, np.where(level, 1, 0))


def _play(table, bracket, home_slot, away_slot, home, away, keys, valid, play_tie):
    """The group stage of scores ``home`` / ``away [n, F]`` ranked once, then the bracket of every simulation.
    ``play_tie(k, home_slot [n], away_slot [n], live [n])`` returns tie k's first or only match ``(home_goals,
    away_goals)``, ``extra [n, 4]`` (as ``settle`` takes it), ``settle``'s verdict ``(A through, how)`` and ``ok``,
    all ``[n]``.  Returns the group stage's ``histograms`` and the bracket's outputs, restricted to the simulations the
    bracket leaves valid."""
    n = len(valid)
    K, nr = len(bracket["round"]), int(bracket["num_rounds"])
    hv, av = np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0)
    pts, gd, gf = tables(table, home_slot, away_slot, hv, av)
    pos = rank(pts, gd, gf, keys, table.get("group"))
    _, sizes = _group_layout(table, int(bracket["num_groups"]))
    qmap, best, ok = qualifiers(table, bracket, pts, gd, gf, keys, np.where(valid[:, None], pos, 0))
    ok &= valid
    kind, a0, a1 = (np.asarray(bracket[k], np.int64) for k in ("kind", "arg0", "arg1"))
    ent = np.zeros((n, K, 2), np.int64)
    ksc = np.zeros((n, K, 2), np.int64)
    kex = np.zeros((n, K, 4), np.int64)
    how = np.zeros((n, K), np.int64)
    win = np.zeros((n, K), np.int64)
    lose = np.zeros((n, K), np.int64)
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
        ksc[:, k, 0], ksc[:, k, 1], kex[:, k], through, how[:, k], tok = play_tie(k, ent[:, k, 0], ent[:, k, 1],
                                                                                 ok.copy())
        ok &= tok
        win[:, k] = np.where(through, ent[:, k, 0], ent[:, k, 1])
        lose[:, k] = np.where(through, ent[:, k, 1], ent[:, k, 0])
    T = len(table["start_points"])
    reach = np.zeros((T, nr), np.int64)
    wins = np.zeros((T, nr), np.int64)
    rnd = np.asarray(bracket["round"], np.int64)
    for k in range(K):
        np.add.at(reach, (win[ok, k], rnd[k]), 1)
        np.add.at(reach, (lose[ok, k], rnd[k]), 1)
        np.add.at(wins, (win[ok, k], rnd[k]), 1)
    bad = ~ok[:, None, None]
    out = histograms(table, pts, pos, ok)
    out.update(ko_entrants=np.where(bad, 255, ent), ko_scores=np.where(bad, 255, ksc),
               ko_winners=np.where(~ok[:, None], 255, win), ko_extra=np.where(bad, 255, kex), reach_counts=reach,
               win_counts=wins, decided_counts=np.stack([np.bincount(how[ok, k], minlength=3)[:3] for k in range(K)]),
               valid=ok, invalid=int((~ok).sum()))
    return out


def resolve_bracket(table, home_slot, away_slot, bracket, home, away, keys, ko_home, ko_away, home_through,
                    valid=None, ko_extra=None):
    """The bracket in pure integer logic from given scores: group scores ``home`` / ``away [n, F]``, tie-break keys
    ``[n, T]``, tie scores ``ko_home`` / ``ko_away [n, K]`` (the first or only match), ``home_through [n, K]`` (whether
    the home entrant won the decider: the lot of a format-0 tie, else the penalties; read only for ties level after
    everything else) and, for ties of format 1 and 2 (``bracket["tie_format"]``), ``ko_extra [n, K, 4]``: leg-2 goals
    of the home and away entrant, then their extra-time goals (read only where that part is played).  Returns
    ``rank_scores``'s outputs restricted to the simulations the bracket leaves valid, ``ko_entrants [n, K, 2]``,
    ``ko_scores``, ``ko_winners [n, K]``, ``ko_extra`` (255 for invalid simulations), ``reach_counts`` / ``win_counts
    [T, rounds]``, ``decided_counts [K, 3]``, ``valid [n]`` and ``invalid``."""
    n = np.asarray(keys).shape[0]
    valid = np.ones(n, bool) if valid is None else np.asarray(valid, bool)
    kh, ka, th = (np.asarray(x).astype(np.int64) for x in (ko_home, ko_away, home_through))
    K = kh.shape[1]
    kx = np.full((n, K, 4), NOT_PLAYED, np.int64) if ko_extra is None else np.asarray(ko_extra, np.int64)
    fmt = _formats(bracket)

    def play(k, hs, as_, live):
        return (kh[:, k], ka[:, k], kx[:, k], *settle(fmt[k], kh[:, k], ka[:, k], kx[:, k], th[:, k].astype(bool)),
                np.ones(n, bool))

    return _play(table, bracket, home_slot, away_slot, np.asarray(home, np.int64), np.asarray(away, np.int64),
                 np.asarray(keys, np.int64), valid, play)


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


def _grid(lh, la, c, G):
    """The normalised clamped, truncated grid ``[n, G + 1, G + 1]`` of ``sample_scores`` (float64)."""
    p, q = _pmf_unnormalised(lh, G), _pmf_unnormalised(la, G)
    w = p[:, :, None] * q[:, None, :]
    w[:, 0, 0] *= np.maximum(1.0 - c * lh * la, 0.0)
    w[:, 0, 1] *= np.maximum(1.0 + c * lh, 0.0)
    w[:, 1, 0] *= np.maximum(1.0 + c * la, 0.0)
    w[:, 1, 1] *= np.maximum(1.0 - c, 0.0)
    return w / w.sum(axis=(1, 2))[:, None, None]


def _goal_difference(w):
    """P(home - away = d), d = -G .. G, ``[n, 2G + 1]``, of grids ``[n, G + 1, G + 1]``."""
    G = w.shape[1] - 1
    return np.stack([np.trace(w, offset=-d, axis1=1, axis2=2) for d in range(-G, G + 1)], axis=1)


def tie_closed_form(model, samples, team_a, team_b, fmt, max_goals, neutral_venue=0, conf_a=0, conf_b=0):
    """Per draw, in float64: ``(P(A through), P(extra time), P(penalties))`` ``[S]`` of one tie of format 1 or 2
    between model teams ``team_a`` (home entrant) and ``team_b``.  The goal difference of the first match (and, for two
    legs, that of leg 2 with the venues swapped, convolved) from each draw's normalised truncated grids, then that of
    extra time (Poisson(lambda / 3) grids of the last match's venue, no tau), then 1/2 for penalties."""
    G = int(max_goals)
    c = np.asarray(samples["corr_coef"], np.float64)
    neutral = model in ("neutral", "neutral_wc")

    def rates(h, a, ch, ca, nv):
        kw = {"home_conf": [ch], "away_conf": [ca]} if model == "neutral_wc" else {}
        if neutral:
            kw["neutral_venue"] = np.array([nv], np.uint8)
        lh, la = op.expected_goals(model, samples, [h], [a], **kw)
        return lh[:, 0], la[:, 0]

    lh, la = rates(team_a, team_b, conf_a, conf_b, neutral_venue)
    d = _goal_difference(_grid(lh, la, c, G))  # A - B
    if fmt == TWO_LEGS:
        lh, la = rates(team_b, team_a, conf_b, conf_a, 0)
        d2 = _goal_difference(_grid(lh, la, c, G))[:, ::-1]  # A - B of leg 2 (A away)
        d = np.stack([np.convolve(x, y) for x, y in zip(d, d2)])
    e = _goal_difference(_grid(lh * EXTRA_TIME_FRACTION, la * EXTRA_TIME_FRACTION, np.zeros_like(c), G))
    if fmt == TWO_LEGS:
        e = e[:, ::-1]
    mid = (d.shape[1] - 1) // 2
    p_level, p_et_level = d[:, mid], e[:, G]
    p_through = d[:, mid + 1:].sum(axis=1) + p_level * (e[:, G + 1:].sum(axis=1) + 0.5 * p_et_level)
    return p_through, p_level, p_level * p_et_level


def simulate_tournament(model, samples, fixtures, home_slot, away_slot, table, bracket, max_goals, sims_per_draw, seed,
                        first_draw=0):
    """The tournaments of draws ``samples`` replayed on the kernel's Philox words: ``resolve_bracket``'s outputs,
    the group stage's ``home`` / ``away`` / ``margin [N, F]`` and ``keys [N, T]`` as ``simulate`` returns them,
    ``ko_margin [N, K]`` (the score walks' margin of the first or only match), ``leg2_margin`` / ``extra_time_margin
    [N, K]`` (those of leg 2 and of extra time where played) and ``decider_margin [N, K]`` (``|u_d (hw + aw) - hw| /
    (hw + aw)`` on drawn format-0 ties, ``|u_d - 1/2|`` on penalties); inf elsewhere."""
    F = 0 if fixtures is None or fixtures.get("home_team") is None else len(fixtures["home_team"])
    T = len(table["start_points"])
    K = len(bracket["round"])
    E = 4 * ((2 * F + T + 3 * K + 3) // 4)
    words, s_of = philox_words(samples, sims_per_draw, seed, first_draw, E + 4 * K)
    N = len(s_of)
    if F:
        home, away, margin, valid = play_fixtures(model, samples, fixtures, home_slot, away_slot, T, max_goals, s_of,
                                                  philox.uniform(words[:, :2 * F]).astype(np.float64))
        home_slot, away_slot = (np.minimum(np.asarray(x, np.int64), T - 1) for x in (home_slot, away_slot))
    else:
        home = away = np.zeros((N, 0), np.int64)
        margin, valid = np.zeros((N, 0)), np.ones(N, bool)
        home_slot = away_slot = np.zeros(0, np.int64)
    keys = words[:, 2 * F:2 * F + T].astype(np.int64)
    u = philox.uniform(words[:, 2 * F + T:2 * F + T + 3 * K]).astype(np.float64)
    ux = philox.uniform(words[:, E:]).astype(np.float64)
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
    nvk = bracket.get("neutral_venue")
    nvk = np.zeros(K, np.int64) if nvk is None else np.asarray(nvk, np.int64)
    ko_margin = np.full((N, K), np.inf)
    leg2_margin = np.full((N, K), np.inf)
    et_margin = np.full((N, K), np.inf)
    dec_margin = np.full((N, K), np.inf)
    fmt = _formats(bracket)

    def play(k, hs, as_, live):
        lh, la = (r[s_of, hs * T + as_] for r in rates[int(nvk[k] and model in ("neutral", "neutral_wc"))])
        h, a, m, v = sample_scores(lh, la, cc, u[:, 3 * k], u[:, 3 * k + 1], max_goals)
        ko_margin[:, k] = np.where(live, m, np.inf)
        extra = np.full((N, 4), NOT_PLAYED, np.int64)
        ud = u[:, 3 * k + 2]
        if fmt[k] == ONE_MATCH:
            hw, aw = win_masses(lh, la, cc, max_goals)
            tot = hw + aw
            drawn = v & (h == a)
            v &= ~drawn | (tot > 0)
            with np.errstate(invalid="ignore", divide="ignore"):
                decider = ud * tot <= hw
                dec_margin[:, k] = np.where(live & drawn, np.abs(ud * tot - hw) / tot, np.inf)
            return h, a, extra, *settle(ONE_MATCH, h, a, extra, decider), v
        ta, tb = h, a
        if fmt[k] == TWO_LEGS:  # leg 2: B at home, never neutral
            lh, la = (r[s_of, as_ * T + hs] for r in rates[0])
            bh, ba, m2, v2 = sample_scores(lh, la, cc, ux[:, 4 * k], ux[:, 4 * k + 1], max_goals)
            leg2_margin[:, k] = np.where(live & v, m2, np.inf)
            v &= v2
            extra[:, 0], extra[:, 1] = ba, bh
            ta, tb = h + ba, a + bh
        level = v & (ta == tb)
        eh, ea, me, ve = sample_scores(lh * EXTRA_TIME_FRACTION, la * EXTRA_TIME_FRACTION, np.zeros(N),
                                       ux[:, 4 * k + 2], ux[:, 4 * k + 3], max_goals)
        et_margin[:, k] = np.where(live & level, me, np.inf)
        v &= ~level | ve
        e_a, e_b = (ea, eh) if fmt[k] == TWO_LEGS else (eh, ea)
        extra[:, 2], extra[:, 3] = np.where(level, e_a, NOT_PLAYED), np.where(level, e_b, NOT_PLAYED)
        pens = level & (ta + e_a == tb + e_b)
        dec_margin[:, k] = np.where(live & pens, np.abs(ud - 0.5), np.inf)
        return h, a, extra, *settle(fmt[k], h, a, extra, ud <= 0.5), v

    out = _play(table, bracket, home_slot, away_slot, home, away, keys, valid, play)
    out.update(home=home, away=away, margin=margin, keys=keys, ko_margin=ko_margin, leg2_margin=leg2_margin,
               extra_time_margin=et_margin, decider_margin=dec_margin)
    return out
