"""Restatement of knockout pairings drawn by lot (``csrc/simulate.cu``, ``simulate_paired_kernel``) in integer and
float64 numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  It builds on ``oracle/tournament.py`` (same group stage, same
ties, same Philox words) and adds the pairings; ``oracle/tournament.py`` itself is the reference of brackets without
them.

Definition (the same text as ``include/bplx.h``): a bracket may carry up to 16 pairings.  Pairing d has a pool of n_d
entrants (SLOT, GROUP_POS, BEST, WINNER, LOSER) and produces n_d / 2 pairs; a tie that takes pair i has entrant kind
PAIRED on both sides, arg0 = d, arg1 = 2i (home) and 2i + 1 (away).  Every pool source is settled before the first tie
that takes a pair of the pairing, and the pairing is made when that tie is reached.  With E = 4 ceil((2F + T_tab +
3K) / 4), pairing d owns Philox blocks ``E/4 + K + 16 d .. + 15``: words w_0 .. w_63, word j = component j mod 4 of
block j / 4.  An index uniform in [0, m) is ``(w m) >> 32``.

* Open: start from pool order p; for i = 0 .. n - 2, j = i + ((w_i (n - i)) >> 32), swap p[i] and p[j].  Pair i =
  (p[2i], p[2i + 1]), the first drawn at home.
* Seeded (pots A and B of equal size <= 16): for pair i, b = the ((w_2i |B left|) >> 32)-th pot-B entrant left in
  pool order; the eligible pot-A entrants left are those b may meet and for which the teams left after removing both
  can still be fully paired; a = the ((w_2i+1 |eligible|) >> 32)-th of them in pool order.  The unseeded entrant is at
  home when the pairing's host pot is 1.  Protections forbid pairs of slots with the same group id (bit 0) or the same
  association (bit 1; 0xFF never clashes).  A pool that cannot be paired at the start makes the simulation invalid.

``open_draw`` and ``seeded_draw`` are the two procedures on given words; ``seeded_pair_proba`` is the exact
distribution of the seeded procedure (a dynamic program over the masks of the entrants left: C(16, 8) = 12,870 states
for 8 + 8), ``uniform_pair_proba`` that of a uniform choice among the valid pairings, which differs from it; an open
draw pairs two given entrants with probability exactly 1 / (n - 1).  ``simulate_tournament`` replays the paired kernel.
"""
from __future__ import annotations

import functools
import itertools

import numpy as np

from oracle import head_to_head as h2h
from oracle import philox
from oracle import tournament as ot
from oracle.simulate import histograms, philox_words, play_fixtures, rank, sample_scores, tables

PAIRED = 5
OPEN, SEEDED = 0, 1
PROTECT_GROUP, PROTECT_ASSOCIATION = 1, 2
MAX_POOL = 64


def index(w, m):
    """An index uniform in [0, m): ``(w m) >> 32``, exact."""
    return (int(w) * int(m)) >> 32


def open_draw(pool, words):
    """Pairs ``[(home, away)]`` of an open draw of ``pool`` (any items) on words ``w_0 ..``."""
    p = list(pool)
    n = len(p)
    for i in range(n - 1):
        j = i + index(words[i], n - i)
        p[i], p[j] = p[j], p[i]
    return [(p[2 * i], p[2 * i + 1]) for i in range(n // 2)]


def _feasible(ra, rb, compat):
    """Whether pot-A entrants ``ra`` and pot-B entrants ``rb`` (index tuples) can be fully paired under ``compat``."""
    match = {}

    def augment(a, seen):
        for b in rb:
            if compat[a][b] and b not in seen:
                seen.add(b)
                if b not in match or augment(match[b], seen):
                    match[b] = a
                    return True
        return False

    return len(ra) == len(rb) and all(augment(a, set()) for a in ra)


def seeded_draw(compat, words):
    """Pairs ``[(a, b)]`` (pot-A index, pot-B index, in draw order) of the seeded procedure on words ``w_0 ..``, with
    ``compat [m][m]`` (a may meet b); None when the pots cannot be fully paired."""
    m = len(compat)
    ra, rb = list(range(m)), list(range(m))
    if not _feasible(ra, rb, compat):
        return None
    pairs = []
    for i in range(m):
        b = rb[index(words[2 * i], len(rb))]
        rb.remove(b)
        elig = [a for a in ra if compat[a][b] and _feasible([x for x in ra if x != a], rb, compat)]
        a = elig[index(words[2 * i + 1], len(elig))]
        ra.remove(a)
        pairs.append((a, b))
    return pairs


def seeded_pair_proba(compat, one=1.0):
    """``[m][m]`` probabilities that the seeded procedure pairs pot-A entrant a with pot-B entrant b (``one``: 1.0
    for float64, ``fractions.Fraction(1)`` for exact values), by a dynamic program over the (A left, B left) masks; None
    when the pots cannot be fully paired."""
    m = len(compat)
    bits = lambda x: [i for i in range(m) if (x >> i) & 1]

    @functools.lru_cache(maxsize=None)
    def feasible(ra, rb):
        return _feasible(bits(ra), bits(rb), compat)

    full = (1 << m) - 1
    if not feasible(full, full):
        return None
    out = [[0 * one for _ in range(m)] for _ in range(m)]
    level = {(full, full): one}
    for _ in range(m):
        nxt = {}
        for (ra, rb), p in level.items():
            bs = bits(rb)
            for b in bs:
                rb2 = rb & ~(1 << b)
                elig = [a for a in bits(ra) if compat[a][b] and feasible(ra & ~(1 << a), rb2)]
                for a in elig:
                    q = p / len(bs) / len(elig)
                    out[a][b] += q
                    key = (ra & ~(1 << a), rb2)
                    nxt[key] = nxt.get(key, 0 * one) + q
        level = nxt
    return out


def uniform_pair_proba(compat, one=1.0):
    """``[m][m]`` pair probabilities of a uniform choice among the valid pairings (every perfect matching equally
    likely): what the sequential procedure is NOT."""
    m = len(compat)
    match = [pm for pm in itertools.permutations(range(m)) if all(compat[a][pm[a]] for a in range(m))]
    out = [[0 * one for _ in range(m)] for _ in range(m)]
    for pm in match:
        for a in range(m):
            out[a][pm[a]] += one / len(match)
    return out


def compat_matrix(slots_a, slots_b, protect, group, assoc):
    """``[m][m]``: pot-A slot a may meet pot-B slot b under the protection bits, the slots' group ids and
    associations (0xFF: none)."""
    def ok(u, v):
        if protect & PROTECT_GROUP and group[u] == group[v]:
            return False
        return not (protect & PROTECT_ASSOCIATION and assoc[u] != 0xFF and assoc[u] == assoc[v])

    return [[ok(u, v) for v in slots_b] for u in slots_a]


def make_pairing(bracket, d, slots, words, group, assoc):
    """Pairing d of one simulation: ``slots`` = its pool resolved to table slots (pool order), ``words`` = its 64
    words.  Returns the pairs ``[(home slot, away slot)]`` in pair order, or None when the pool cannot be paired."""
    if int(bracket["pairing_mode"][d]) == OPEN:
        return open_draw(slots, words)
    pots = np.asarray(bracket["pool_pot"])[d, :len(slots)]
    sa = [s for s, p in zip(slots, pots) if p == 0]
    sb = [s for s, p in zip(slots, pots) if p == 1]
    prot = int(bracket["pairing_protect"][d]) if bracket.get("pairing_protect") is not None else 0
    pairs = seeded_draw(compat_matrix(sa, sb, prot, group, assoc), words)
    if pairs is None:
        return None
    unseeded_home = bracket.get("pairing_host_pot") is not None and int(bracket["pairing_host_pot"][d])
    return [(sb[b], sa[a]) if unseeded_home else (sa[a], sb[b]) for a, b in pairs]


def _pairing_ties(bracket):
    """``first [P]`` (the tie at which pairing d is made) and ``of_tie [K]`` ((d, i) of the pair tie k takes, or
    None)."""
    kind, a0, a1 = (np.asarray(bracket[k], np.int64) for k in ("kind", "arg0", "arg1"))
    of_tie, first = [], {}
    for k in range(len(kind)):
        if kind[k, 0] == PAIRED:
            d = int(a0[k, 0])
            of_tie.append((d, int(a1[k, 0]) // 2))
            first.setdefault(d, k)
        else:
            of_tie.append(None)
    return first, of_tie


def simulate_tournament(model, samples, fixtures, home_slot, away_slot, table, bracket, max_goals, sims_per_draw, seed,
                        first_draw=0, tiebreak="goal_difference", played_h2h=None):
    """The tournaments of draws ``samples`` with the pairings of ``bracket`` (``season.build_bracket``) replayed on the
    kernel's Philox words: ``oracle.tournament.simulate_tournament``'s outputs (the group ranked under ``tiebreak``)
    plus ``pairing_counts [P, T, T]``; ``small_margin [N]`` marks simulations where some score walk or decider is at
    rounding level (the float32 kernel may differ from this replay only there)."""
    F = 0 if fixtures is None or fixtures.get("home_team") is None else len(fixtures["home_team"])
    T = len(table["start_points"])
    K = len(bracket["round"])
    P = len(bracket["pool_size"])
    E = 4 * ((2 * F + T + 3 * K + 3) // 4)
    P0 = E // 4 + K
    words, s_of = philox_words(samples, sims_per_draw, seed, first_draw, 4 * (P0 + 16 * P))
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
    ux = philox.uniform(words[:, E:E + 4 * K]).astype(np.float64)
    pw = words[:, 4 * P0:].astype(np.int64)  # [N, 64 P]
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
            rates[nv] = ot.op.expected_goals(model, samples, ht, at, **extra)
    cc = np.asarray(samples["corr_coef"], np.float64)[s_of]
    nvk = bracket.get("neutral_venue")
    nvk = np.zeros(K, np.int64) if nvk is None else np.asarray(nvk, np.int64)
    fmt = ot._formats(bracket)
    small = np.zeros(N, bool)
    tiny = 1e-5

    def play(k, hs, as_, live):
        """One tie (``oracle.tournament.simulate_tournament``'s), marking rounding-level margins in ``small``."""
        nonlocal small
        lh, la = (r[s_of, hs * T + as_] for r in rates[int(nvk[k] and model in ("neutral", "neutral_wc"))])
        h, a, m, v = sample_scores(lh, la, cc, u[:, 3 * k], u[:, 3 * k + 1], max_goals)
        small |= live & (m < tiny)
        extra = np.full((N, 4), ot.NOT_PLAYED, np.int64)
        ud = u[:, 3 * k + 2]
        if fmt[k] == ot.ONE_MATCH:
            hw, aw = ot.win_masses(lh, la, cc, max_goals)
            tot = hw + aw
            drawn = v & (h == a)
            v &= ~drawn | (tot > 0)
            with np.errstate(invalid="ignore", divide="ignore"):
                decider = ud * tot <= hw
                small |= live & drawn & (np.abs(ud * tot - hw) / tot < tiny)
            return h, a, extra, *ot.settle(ot.ONE_MATCH, h, a, extra, decider), v
        ta, tb = h, a
        if fmt[k] == ot.TWO_LEGS:
            lh, la = (r[s_of, as_ * T + hs] for r in rates[0])
            bh, ba, m2, v2 = sample_scores(lh, la, cc, ux[:, 4 * k], ux[:, 4 * k + 1], max_goals)
            small |= live & v & (m2 < tiny)
            v &= v2
            extra[:, 0], extra[:, 1] = ba, bh
            ta, tb = h + ba, a + bh
        level = v & (ta == tb)
        eh, ea, me, ve = sample_scores(lh * ot.EXTRA_TIME_FRACTION, la * ot.EXTRA_TIME_FRACTION, np.zeros(N),
                                       ux[:, 4 * k + 2], ux[:, 4 * k + 3], max_goals)
        small |= live & level & (me < tiny)
        v &= ~level | ve
        e_a, e_b = (ea, eh) if fmt[k] == ot.TWO_LEGS else (eh, ea)
        extra[:, 2], extra[:, 3] = np.where(level, e_a, ot.NOT_PLAYED), np.where(level, e_b, ot.NOT_PLAYED)
        pens = level & (ta + e_a == tb + e_b)
        small |= live & pens & (np.abs(ud - 0.5) < tiny)
        return h, a, extra, *ot.settle(fmt[k], h, a, extra, ud <= 0.5), v

    # the group stage ranked once, then the bracket (oracle.tournament._play, with the pairings)
    n = N
    nr = int(bracket["num_rounds"])
    hv, av = np.where(valid[:, None], home, 0), np.where(valid[:, None], away, 0)
    pts, gd, gf = tables(table, home_slot, away_slot, hv, av)
    if tiebreak == "head_to_head":
        pos = h2h.rank(table, home_slot, away_slot, hv, av, keys, played_h2h)
    else:
        pos = rank(pts, gd, gf, keys, table.get("group"))
    _, sizes = ot._group_layout(table, int(bracket["num_groups"]))
    qmap, best, ok = ot.qualifiers(table, bracket, pts, gd, gf, keys, np.where(valid[:, None], pos, 0))
    ok &= valid
    kind, a0, a1 = (np.asarray(bracket[x], np.int64) for x in ("kind", "arg0", "arg1"))
    group = np.zeros(T, np.int64) if table.get("group") is None else np.asarray(table["group"], np.int64)
    assoc = np.full(T, 0xFF, np.int64) if bracket.get("slot_assoc") is None else np.asarray(bracket["slot_assoc"],
                                                                                             np.int64)
    first, of_tie = _pairing_ties(bracket)
    drawn = {}  # (d, i) -> ([n] home, [n] away)
    ent = np.zeros((n, K, 2), np.int64)
    ksc = np.zeros((n, K, 2), np.int64)
    kex = np.zeros((n, K, 4), np.int64)
    how = np.zeros((n, K), np.int64)
    win = np.zeros((n, K), np.int64)
    lose = np.zeros((n, K), np.int64)

    def source(kd, x, y):
        nonlocal ok
        if kd == ot.SLOT:
            return np.full(n, x)
        if kd == ot.GROUP_POS:
            inside = y < sizes[x]
            ok &= inside
            return qmap[:, x, y] if inside else np.zeros(n, np.int64)
        if kd == ot.BEST:
            return best[:, x]
        return win[:, x] if kd == ot.WINNER else lose[:, x]

    for k in range(K):
        for d, kf in first.items():
            if kf != k:
                continue
            size = int(bracket["pool_size"][d])
            pool = np.stack([source(*(int(bracket[x][d, j]) for x in ("pool_kind", "pool_arg0", "pool_arg1")))
                             for j in range(size)], axis=1)
            hh, aa = np.zeros((n, size // 2), np.int64), np.zeros((n, size // 2), np.int64)
            for i in np.flatnonzero(ok):
                pairs = make_pairing(bracket, d, pool[i].tolist(), pw[i, 64 * d:64 * d + 64], group, assoc)
                if pairs is None:
                    ok[i] = False
                    continue
                hh[i], aa[i] = [p[0] for p in pairs], [p[1] for p in pairs]
            for i in range(size // 2):
                drawn[(d, i)] = (hh[:, i], aa[:, i])
        if of_tie[k] is not None:
            for side in range(2):
                ent[:, k, side] = np.where(ok, drawn[of_tie[k]][side], 0)
        else:
            for side in range(2):
                ent[:, k, side] = np.where(ok, source(kind[k, side], a0[k, side], a1[k, side]), 0)
        ksc[:, k, 0], ksc[:, k, 1], kex[:, k], through, how[:, k], tok = play(k, ent[:, k, 0], ent[:, k, 1], ok.copy())
        ok &= tok
        win[:, k] = np.where(through, ent[:, k, 0], ent[:, k, 1])
        lose[:, k] = np.where(through, ent[:, k, 1], ent[:, k, 0])
    reach = np.zeros((T, nr), np.int64)
    wins = np.zeros((T, nr), np.int64)
    pc = np.zeros((P, T, T), np.int64)
    rnd = np.asarray(bracket["round"], np.int64)
    for k in range(K):
        np.add.at(reach, (win[ok, k], rnd[k]), 1)
        np.add.at(reach, (lose[ok, k], rnd[k]), 1)
        np.add.at(wins, (win[ok, k], rnd[k]), 1)
        if of_tie[k] is not None:
            np.add.at(pc, (of_tie[k][0], ent[ok, k, 0], ent[ok, k, 1]), 1)
    bad = ~ok[:, None, None]
    out = histograms(table, pts, pos, ok)
    out.update(ko_entrants=np.where(bad, 255, ent), ko_scores=np.where(bad, 255, ksc),
               ko_winners=np.where(~ok[:, None], 255, win), ko_extra=np.where(bad, 255, kex), reach_counts=reach,
               win_counts=wins, decided_counts=np.stack([np.bincount(how[ok, k], minlength=3)[:3] for k in range(K)]),
               pairing_counts=pc, valid=ok, invalid=int((~ok).sum()), home=home, away=away, margin=margin, keys=keys,
               small_margin=small | (margin < tiny).any(axis=1))
    return out
