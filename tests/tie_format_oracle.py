"""Knockout tie formats restated in float64 numpy, on top of ``tests/tournament_oracle.py``.

TEST INFRASTRUCTURE ONLY.  ``tournament_oracle`` restates the group stage and the bracket of one-match ties (format 0);
this module adds a format byte per tie (``bracket["tie_format"]``, all 0 when absent), with the definition of
``include/bplx.h``:

  0 BPLX_TIE_ONE_MATCH     one match; a draw is decided by ``u_d (hw + aw) <= hw``
  1 BPLX_TIE_ONE_MATCH_ET  one match; drawn: extra time; still level: penalties
  2 BPLX_TIE_TWO_LEGS      two legs; level on aggregate: extra time in leg 2; still level: penalties

The home entrant A hosts leg 1, the away entrant B leg 2 with the venues swapped (neutral_venue 0 in both legs; for
NeutralWC the confederations swap sides); each leg is a 90-minute match sampled like a group fixture.  Aggregate
``A = h1 + a2``, ``B = a1 + h2``; the higher goes through, no away-goals rule.  Extra time is played at the venue of the
last match (format 1: with the tie's neutral flag) on the draw's rates times ``EXTRA_TIME_FRACTION = 1/3``, without the
tau correction (independent Poissons truncated at G).  Penalties: A goes through iff ``u_d <= 1/2``.  Tie k keeps words
``2F + T_tab + 3k .. + 2``; with ``E = 4 ceil((2F + T_tab + 3K) / 4)`` it owns words ``E + 4k .. E + 4k + 3``: leg 2
``(u_h, u_a)``, then extra time ``(u_h, u_a)``.  A non-finite rate or normaliser in leg 2 or in extra time makes the
simulation invalid, as in the first match.

``resolve_bracket`` is the bracket in pure integer logic from given scores and decider outcomes; ``simulate_tournament``
replays the kernel on the same Philox words and returns a per-tie margin for the score walks of every match and for
the decider (``|u_d (hw + aw) - hw| / (hw + aw)``, or ``|u_d - 1/2|`` for penalties): the float32 kernel may differ
from it only where a margin is at rounding level.  ``tie_closed_form`` gives, per draw, P(A through), P(extra time) and
P(penalties) of one tie between two fixed teams by convolving goal-difference distributions.  Both reuse
``tournament_oracle``'s bracket walk (entrants, qualifiers, winners, reach / win counts) unchanged.
"""
from __future__ import annotations

import numpy as np

from oracle import philox
from oracle import predict as op
from oracle.simulate import _pmf_unnormalised, rank, rank_scores, sample_scores, simulate, tables
from tests.tournament_oracle import _play_bracket, win_masses

ONE_MATCH, ONE_MATCH_ET, TWO_LEGS = 0, 1, 2
EXTRA_TIME_FRACTION = 1.0 / 3.0
NOT_PLAYED = 254


def _formats(bracket):
    K = len(bracket["round"])
    f = bracket.get("tie_format")
    return np.zeros(K, np.int64) if f is None else np.asarray(f, np.int64)


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


def _play_formats(table, bracket, pts, gd, gf, keys, pos, valid, play_tie):
    """``tournament_oracle._play_bracket`` with tie formats: ``play_tie(k, home_slot [n], away_slot [n], live [n])``
    returns ``(home_goals, away_goals, extra [n, 4], decider [n], ok)`` for tie k (``settle``'s inputs).  The walk is
    handed level scores and ``settle``'s verdict, so it takes each winner from the verdict; the real scores, ``extra``
    and how each tie was settled are kept here.  Adds ``ko_extra [n, K, 4]`` and ``decided_counts [K, 3]``."""
    n, K = pos.shape[0], len(bracket["round"])
    fmt = _formats(bracket)
    ksc = np.zeros((n, K, 2), np.int64)
    kex = np.full((n, K, 4), NOT_PLAYED, np.int64)
    how = np.zeros((n, K), np.int64)
    level = np.zeros(n, np.int64)

    def play(k, hs, as_, live):
        h, a, extra, decider, ok = play_tie(k, hs, as_, live)
        ksc[:, k, 0], ksc[:, k, 1] = h, a
        kex[:, k] = extra
        through, how[:, k] = settle(fmt[k], h, a, extra, decider)
        return level, level, through, ok

    out = _play_bracket(table, bracket, pts, gd, gf, keys, pos, valid, play)
    ok = out["valid"]
    bad = ~ok[:, None, None]
    out.update(ko_scores=np.where(bad, 255, ksc), ko_extra=np.where(bad, 255, kex),
               decided_counts=np.stack([np.bincount(how[ok, k], minlength=3)[:3] for k in range(K)]))
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
    home, away = np.asarray(home, np.int64), np.asarray(away, np.int64)
    hv, av = np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0)
    pts, gd, gf = tables(table, home_slot, away_slot, hv, av)
    keys = np.asarray(keys, np.int64)
    pos = rank(pts, gd, gf, keys, table.get("group"))
    kh, ka, th = (np.asarray(x).astype(np.int64) for x in (ko_home, ko_away, home_through))
    K = kh.shape[1]
    kx = np.full((n, K, 4), NOT_PLAYED, np.int64) if ko_extra is None else np.asarray(ko_extra, np.int64)

    def play(k, hs, as_, live):
        return kh[:, k], ka[:, k], kx[:, k], th[:, k].astype(bool), np.ones(n, bool)

    out = _play_formats(table, bracket, pts, gd, gf, keys, pos, valid, play)
    r = rank_scores(table, home_slot, away_slot, home, away, keys, out["valid"])
    out.update(r, invalid=int((~out["valid"]).sum()))
    return out


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
    """The tournaments of draws ``samples`` replayed on the kernel's Philox words: ``simulate``'s outputs for the
    group stage plus ``_play_formats``'s, ``ko_margin [N, K]`` (the score walks' margin of the first or only match),
    ``leg2_margin`` / ``extra_time_margin [N, K]`` (those of leg 2 and of extra time where played) and
    ``decider_margin [N, K]`` (``|u_d (hw + aw) - hw| / (hw + aw)`` on drawn format-0 ties, ``|u_d - 1/2|`` on
    penalties); inf elsewhere."""
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
    E = 4 * ((2 * F + T + 3 * K + 3) // 4)
    words = philox.stream(int(seed), n_glob.astype(np.uint64), 0, E + 4 * K)
    keys = words[:, 2 * F:2 * F + T].astype(np.int64)
    u = philox.uniform(words[:, 2 * F + T:2 * F + T + 3 * K]).astype(np.float64)
    ux = philox.uniform(words[:, E:]).astype(np.float64)
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
                through = ud * tot <= hw
                dec_margin[:, k] = np.where(live & drawn, np.abs(ud * tot - hw) / tot, np.inf)
            return h, a, extra, through, v
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
        return h, a, extra, ud <= 0.5, v

    out = _play_formats(table, bracket, pts, gd, gf, keys, pos, valid, play)
    r = rank_scores(table, np.minimum(home_slot, T - 1), np.minimum(away_slot, T - 1), g["home"], g["away"], keys,
                    out["valid"])
    out.update(r, home=g["home"], away=g["away"], margin=g["margin"], keys=keys, ko_margin=ko_margin,
               leg2_margin=leg2_margin, extra_time_margin=et_margin, decider_margin=dec_margin,
               invalid=int((~out["valid"]).sum()))
    return out
