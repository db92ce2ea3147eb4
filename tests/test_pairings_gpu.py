"""Pairings drawn by lot on the GPU: brackets without pairings through the paired entry point bit-identical to
bplx_simulate_tournament_ranked, the paired kernel replayed by the float64 / integer reference (oracle/pairing.py)
for all four models, draw ranges and seeds, the distribution of seeded and open draws against their exact
probabilities, pools that cannot be paired, the UEFA-shaped competition through the predictor, and refusals."""
import numpy as np
import pytest

from bpl_next_b200 import _abi, problem, season
from oracle import pairing as op
from tests import test_head_to_head_gpu as th
from tests import test_tournament_gpu as ttour
from tests.test_pairings import protected_8_8
from tests.test_score_grid_gpu import make_samples
from tests.test_simulate_gpu import _dev

pytestmark = pytest.mark.gpu

MODELS = ["dixon_coles", "extended", "neutral", "neutral_wc"]


def _run(model, s, fx, hs, as_, tab, br, R, seed, first_draw=0, raw=True):
    from bpl_next_b200 import simulate_tournament

    dfx = _dev(dict(fx, home_slot=hs, away_slot=as_)) if len(hs) else {}
    out = simulate_tournament(model, _dev(s), dfx, th._dev_table(tab), br, 15, R, seed, first_draw=first_draw,
                              want_positions=raw, want_scores=raw, want_knockout=raw)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def test_no_pairings_through_the_paired_entry_point_is_bitwise_ranked(monkeypatch):
    """The 48-team World Cup shape under both ranking rules: every output of the paired call with zero pairings equals
    bplx_simulate_tournament_ranked's."""
    s, fx, hs, as_, tab, br = ttour._case("neutral_wc", 37, 48, True, 72, seed=81, best=True)
    for rule in ("goal_difference", "head_to_head"):
        t = dict(tab, tiebreak=rule, played_h2h=th._played(48, 2) if rule == "head_to_head" else None)
        old = _run("neutral_wc", s, fx, hs, as_, t, br, 4, seed=13)
        with monkeypatch.context() as mp:
            mp.setattr(problem, "_pairings_struct", lambda b, T, keep: _abi.Pairings())
            new = _run("neutral_wc", s, fx, hs, as_, t, br, 4, seed=13)
        assert set(new) == set(old) | {"pairing_counts"} and new["pairing_counts"].shape == (0, 48, 48)
        for k in old:
            if old[k] is not None:
                np.testing.assert_array_equal(old[k], new[k], err_msg=f"{rule} {k}")


def _paired_case(model, S, F, seed, Cf=4):
    """16 slots in 4 groups of 4 and F random fixtures; a seeded quarter-final of the group winners against the
    runners-up (group protection, and association protection with a few slots sharing associations), two-legged and
    with extra time; an open semi-final draw of the four winners (extra time); a final (one match) and a third-place
    match (two legs) between fixed winners and losers."""
    s, fx, hs, as_, tab, br0 = ttour._case(model, S, 16, True, F, seed, Cf=Cf)
    L = tab["group_labels"]
    pairings = [{"id": "qf", "pool": [("group", g, 0) for g in L] + [("group", g, 1) for g in L],
                 "pots": [0] * 4 + [1] * 4, "protect": {"group", "association"}, "seeded_home": seed % 2 == 0},
                {"id": "sf", "pool": [("winner", f"qf{i}") for i in range(4)], "pots": None}]
    fmts = ["two_legs", "extra_time", "one_match", "two_legs"]
    ties = [{"id": f"qf{i}", "round": "QF", "pair": ("qf", i), "format": fmts[i]} for i in range(4)]
    ties += [{"id": f"sf{i}", "round": "SF", "pair": ("sf", i), "format": "extra_time"} for i in range(2)]
    ties += [{"id": "third", "round": "3rd", "home": ("loser", "sf0"), "away": ("loser", "sf1"), "format": "two_legs"},
             {"id": "final", "round": "F", "home": ("winner", "sf0"), "away": ("winner", "sf1")}]
    assoc = {f"S{i}": a for i, a in zip(range(16), [0, 1, 2, 3, 0, 1, 2, 3, None, 1, 0, 2, 0, None, 3, 1])}
    br = season.build_bracket(tab, ties, pairings=pairings, association=assoc)
    br["slot_team"] = br0["slot_team"]
    if model == "neutral_wc":
        br["slot_conf"] = br0["slot_conf"]
    return s, fx, hs, as_, tab, br


RAW = ("positions", "ko_entrants", "ko_winners", "ko_extra", "ko_scores")
COUNTS = ("position_counts", "points_counts", "reach_counts", "win_counts", "decided_counts", "pairing_counts")


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("tiebreak", ["goal_difference", "head_to_head"])
def test_exact_replay(model, tiebreak):
    """Raw rows equal the reference's replay on the same Philox words except in simulations where a score walk or
    decider is at rounding level (at most 1 %), and every count equals the reference's when no row differs."""
    S, R, seed = 61, 3, 5000 + len(model) + len(tiebreak)
    s, fx, hs, as_, tab, br = _paired_case(model, S, 40, seed)
    if tiebreak == "head_to_head":
        tab = dict(tab, tiebreak="head_to_head", played_h2h=th._played(16, seed))
    k = _run(model, s, fx, hs, as_, tab, br, R, seed)
    o = op.simulate_tournament(model, s, fx, hs, as_, tab, br, 15, R, seed, tiebreak=tiebreak,
                               played_h2h=tab.get("played_h2h"))
    n = len(o["valid"])
    differ = np.zeros(n, bool)
    for key in RAW:
        differ |= (k[key].astype(np.int64) != o[key]).reshape(n, -1).any(axis=1)
    assert not (differ & ~o["small_margin"]).any(), np.flatnonzero(differ & ~o["small_margin"])[:5]
    assert differ.mean() <= 0.01
    if not differ.any():
        assert k["invalid"][0] == o["invalid"]
        for key in COUNTS:
            np.testing.assert_array_equal(k[key], o[key], err_msg=key)
    # the drawn quarter-finals respect the protections, and some simulations draw differently
    ent = k["ko_entrants"][k["ko_winners"][:, 0] != 0xFF, :4].astype(np.int64)
    grp, assoc = np.asarray(tab["group"]), br["slot_assoc"]
    assert not (grp[ent[:, :, 0]] == grp[ent[:, :, 1]]).any()
    a0, a1 = assoc[ent[:, :, 0]], assoc[ent[:, :, 1]]
    assert not ((a0 == a1) & (a0 != 0xFF)).any()
    assert len({tuple(r) for r in ent.reshape(len(ent), -1)}) > 10


def test_draw_ranges_and_seeds():
    s, fx, hs, as_, tab, br = _paired_case("neutral", 40, 40, seed=8)
    full = _run("neutral", s, fx, hs, as_, tab, br, 4, seed=3)
    parts = [_run("neutral", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, br, 4, seed=3, first_draw=lo)
             for lo, hi in ((0, 13), (13, 40))]
    for key in COUNTS:
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key], err_msg=key)
    for key in RAW:
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]), err_msg=key)
    other = _run("neutral", s, fx, hs, as_, tab, br, 4, seed=4)
    assert not np.array_equal(full["pairing_counts"], other["pairing_counts"])
    noraw = _run("neutral", s, fx, hs, as_, tab, br, 4, seed=3, raw=False)
    np.testing.assert_array_equal(full["pairing_counts"], noraw["pairing_counts"])


def _cup(S, pairings, ties, names, groups=None, association=None):
    tab = season.build_table(names, groups=groups)
    season._size_histograms(tab)
    br = season.build_bracket(tab, ties, pairings=pairings, association=association)
    br["slot_team"] = np.arange(len(names), dtype=np.uint16)
    return make_samples("dixon_coles", S, len(names), 4, seed=S), tab, br


def _within(k, p, N, what):
    sigma = np.sqrt(p * (1 - p) / N)
    bad = np.abs(k / N - p) > 5 * sigma + 1e-12
    assert not bad.any(), (what, np.argwhere(bad)[:5], (k / N)[bad][:5], np.asarray(p)[bad][:5])


def test_seeded_distribution_against_the_exact_procedure():
    """A seeded 8 + 8 pool with group and association protection (F = 0, fixed slots), N = 2^22: every pair
    probability within 5 sigma of the dynamic program's, forbidden pairs never drawn, the unseeded team always at
    home."""
    group, assoc, compat = protected_8_8()
    names = [f"W{g}" for g in range(8)] + [f"R{g}" for g in range(8)]
    pairings = [{"id": "r16", "pool": [("team", n) for n in names], "pots": [0] * 8 + [1] * 8,
                 "protect": {"group", "association"}, "seeded_home": False}]
    ties = [{"id": f"t{i}", "round": "R16", "pair": ("r16", i)} for i in range(8)]
    prev = [f"t{i}" for i in range(8)]
    while len(prev) > 1:
        nxt = [f"{prev[j]}+" for j in range(0, len(prev), 2)]
        ties += [{"id": nxt[j // 2], "round": f"r{len(prev)}", "home": ("winner", prev[j]),
                  "away": ("winner", prev[j + 1])} for j in range(0, len(prev), 2)]
        prev = nxt
    S, R = 64, 65536
    N = S * R
    s, tab, br = _cup(S, pairings, ties, names, groups=[f"g{g}" for g in group],
                      association=[None if a == 0xFF else a for a in assoc])
    k = _run("dixon_coles", s, {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8), tab, br, R, seed=11, raw=False)
    assert k["invalid"][0] == 0
    pc = k["pairing_counts"][0]
    dp = np.array(op.seeded_pair_proba(compat))
    _within(pc[8:, :8].T, dp, N, "seeded")
    assert (pc[:8, :] == 0).all() and (pc[8:, 8:] == 0).all()  # the unseeded team is at home; no pot meets itself
    assert (pc[8:, :8].T[~np.array(compat)] == 0).all()
    assert pc.sum() == 8 * N


def test_open_distribution():
    """An open draw of 16 (F = 0), N = 2^22: every unordered pair within 5 sigma of 1/15, every ordered pair of 1/30,
    and every team at home within 5 sigma of 1/2."""
    names = [f"S{i}" for i in range(16)]
    pairings = [{"id": "r1", "pool": [("team", n) for n in names], "pots": None}]
    ties = [{"id": f"t{i}", "round": "R1", "pair": ("r1", i)} for i in range(8)]
    prev = [f"t{i}" for i in range(8)]
    while len(prev) > 1:
        nxt = [f"{prev[j]}+" for j in range(0, len(prev), 2)]
        ties += [{"id": nxt[j // 2], "round": f"r{len(prev)}", "home": ("winner", prev[j]),
                  "away": ("winner", prev[j + 1])} for j in range(0, len(prev), 2)]
        prev = nxt
    S, R = 64, 65536
    N = S * R
    s, tab, br = _cup(S, pairings, ties, names)
    k = _run("dixon_coles", s, {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8), tab, br, R, seed=12, raw=False)
    assert k["invalid"][0] == 0
    pc = k["pairing_counts"][0]
    off = ~np.eye(16, dtype=bool)
    assert (np.diag(pc) == 0).all()
    _within((pc + pc.T)[off], np.full(off.sum(), 1 / 15), N, "unordered")
    _within(pc[off], np.full(off.sum(), 1 / 30), N, "ordered")
    _within(pc.sum(axis=1), np.full(16, 0.5), N, "home")


def test_pools_that_cannot_be_paired_are_invalid():
    """A seeded pool of group-stage entrants under association protection that some group results leave unpairable:
    those simulations are counted in `invalid`, their raw rows are 0xFF, and no histogram counts them; the reference
    agrees simulation by simulation."""
    s, fx, hs, as_, tab, br0 = ttour._case("dixon_coles", 101, 8, True, 24, seed=91)
    L = tab["group_labels"]
    pairings = [{"id": "sf", "pool": [("group", L[0], 0), ("group", L[1], 0), ("group", L[0], 1), ("group", L[1], 1)],
                 "pots": [0, 0, 1, 1], "protect": {"association"}}]
    ties = [{"id": "s0", "round": "SF", "pair": ("sf", 0)}, {"id": "s1", "round": "SF", "pair": ("sf", 1)},
            {"id": "f", "round": "F", "home": ("winner", "s0"), "away": ("winner", "s1")}]
    assoc = ["x", "x", None, None, "x", "x", None, None]  # the top two of either group can clash
    br = season.build_bracket(tab, ties, pairings=pairings, association=assoc)
    br["slot_team"] = br0["slot_team"]
    k = _run("dixon_coles", s, fx, hs, as_, tab, br, 5, seed=2)
    N = 101 * 5
    bad = k["ko_winners"][:, 0] == 0xFF
    assert 0 < k["invalid"][0] == bad.sum() < N
    assert (k["ko_entrants"][bad] == 0xFF).all() and (k["positions"][bad] == 0xFF).all()
    valid = N - int(k["invalid"][0])
    assert k["pairing_counts"].sum() == 2 * valid and k["win_counts"].sum() == 3 * valid
    assert k["position_counts"].sum() == 8 * valid
    o = op.simulate_tournament("dixon_coles", s, fx, hs, as_, tab, br, 15, 5, seed=2)
    clean = ~o["small_margin"]
    np.testing.assert_array_equal(bad[clean], ~o["valid"][clean])


def test_uefa_shaped_competition_end_to_end():
    """32 teams in 8 groups of four (head-to-head), a seeded round of 16 under group and association protection,
    open quarter- and semi-final draws, all two-legged, and a final, through the predictor: each team's share of a
    draw's pairs is its probability of being in the pool, and the round after a draw is reached by its ties'
    winners."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor

    m = ttour._wc_predictor(S=128)
    teams = [f"T{i:02d}" for i in range(32)]
    L = "ABCDEFGH"
    groups = {t: L[i // 4] for i, t in enumerate(teams)}
    conf = {t: f"C{i % 6}" for i, t in enumerate(teams)}
    pairs = [(teams[4 * g + i], teams[4 * g + j]) for g in range(8) for i in range(4) for j in range(4) if i != j]
    fx = {"home_team": [a for a, _ in pairs], "away_team": [b for _, b in pairs],
          "home_conf": [conf[a] for a, _ in pairs], "away_conf": [conf[b] for _, b in pairs],
          "neutral_venue": [0] * len(pairs)}
    pairings = [{"id": "r16", "pool": [("group", g, 0) for g in L] + [("group", g, 1) for g in L],
                 "pots": [0] * 8 + [1] * 8, "protect": {"group", "association"}},
                {"id": "qf", "pool": [("winner", f"r16_{i}") for i in range(8)], "pots": None},
                {"id": "sf", "pool": [("winner", f"qf_{i}") for i in range(4)], "pots": None}]
    ties = [{"id": f"r16_{i}", "round": "R16", "pair": ("r16", i), "format": "two_legs"} for i in range(8)]
    ties += [{"id": f"qf_{i}", "round": "QF", "pair": ("qf", i), "format": "two_legs"} for i in range(4)]
    ties += [{"id": f"sf_{i}", "round": "SF", "pair": ("sf", i), "format": "two_legs"} for i in range(2)]
    ties += [{"id": "final", "round": "F", "home": ("winner", "sf_0"), "away": ("winner", "sf_1"),
              "format": "extra_time", "neutral_venue": 1}]
    assoc = {t: f"N{i // 8}" for i, t in enumerate(teams)}  # two groups per association: always pairable
    res = m.simulate_tournament(fx, ties, groups=groups, num_sims_per_draw=16, random_state=5, tiebreak="head_to_head",
                                pairings=pairings, association=assoc)
    assert res["pairing_ids"] == ["r16", "qf", "sf"] and res["pairing_proba"].shape == (3, 32, 32)
    pp, pos, win, reach = res["pairing_proba"], res["position_proba"], res["win_proba"], res["reach_proba"]
    share = pp.sum(axis=2) + pp.sum(axis=1)  # [3, T]
    np.testing.assert_allclose(share[0], pos[:, 0] + pos[:, 1], rtol=0, atol=1e-12)
    np.testing.assert_allclose(share[1], win[:, 0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(share[2], win[:, 1], rtol=0, atol=1e-12)
    for r in range(3):
        np.testing.assert_allclose(reach[:, r + 1], win[:, r], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res["champion_proba"].sum(), 1.0, rtol=0, atol=1e-12)
    # protections hold: no pair of the same group, nor of the same association
    g = np.array([L.index(groups[t]) for t in teams])
    a = np.array([int(assoc[t][1:]) for t in teams])
    same = (g[:, None] == g[None, :]) | (a[:, None] == a[None, :])
    assert (pp[0][same] == 0).all()
    # the unseeded runner-up is at home in leg 1: a team is at home in the round of 16 iff it was second
    np.testing.assert_allclose(pp[0].sum(axis=1), pos[:, 1], rtol=0, atol=1e-12)
    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().simulate_tournament(fx, ties, pairings=pairings)


def _refused(br, tab, status=_abi.E_INVALID, match=None):
    s = make_samples("dixon_coles", 4, 16, 4, seed=1)
    with pytest.raises(_abi.BplxError, match=match) as e:
        _run("dixon_coles", s, {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8), tab, br, 2, seed=1)
    assert e.value.status == status


def test_refusals():
    names = [f"S{i}" for i in range(16)]
    tab = season.build_table(names, groups=[f"g{i // 4}" for i in range(16)])
    season._size_histograms(tab)
    pairings = [{"id": "a", "pool": [("team", n) for n in names[:8]], "pots": [0] * 4 + [1] * 4,
                 "protect": {"group"}},
                {"id": "b", "pool": [("winner", f"a{i}") for i in range(4)], "pots": None}]
    ties = [{"id": f"a{i}", "round": "R1", "pair": ("a", i)} for i in range(4)]
    ties += [{"id": f"b{i}", "round": "R2", "pair": ("b", i)} for i in range(2)]
    ties += [{"id": "f", "round": "F", "home": ("winner", "b0"), "away": ("winner", "b1")}]
    good = season.build_bracket(tab, ties, pairings=pairings)
    good["slot_team"] = np.arange(16, dtype=np.uint16)
    s = make_samples("dixon_coles", 4, 16, 4, seed=1)
    ok = _run("dixon_coles", s, {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8), tab, good, 2, seed=1)
    assert ok["invalid"][0] == 0

    def bad(**kv):
        b = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in good.items()}
        for k, f in kv.items():
            f(b[k])
        return b

    def setv(idx, v):
        def f(a):
            a[idx] = v
        return f

    _refused(bad(pool_size=setv(1, 5)), tab, match="even size")  # an odd open pool
    _refused(bad(pool_size=setv(1, 66)), tab, match="even size")  # an open pool above 64
    _refused(bad(pool_pot=setv((0, 0), 1)), tab, match="pots differ")  # unequal pots
    big = bad(pool_size=setv(0, 34), pool_pot=setv((0, slice(0, 34)), [0] * 17 + [1] * 17),
              pool_kind=setv((0, slice(0, 34)), _abi.ENTRANT_SLOT), pool_arg0=setv((0, slice(0, 34)), 0))
    _refused(big, tab, match="at most 16")  # pots above 16
    _refused(bad(pairing_protect=setv(1, 1)), tab, match="seeded")  # protection on an open pairing
    _refused(bad(pool_kind=setv((1, 0), _abi.ENTRANT_PAIRED)), tab, match="inside a pool")
    _refused(bad(pool_arg0=setv((1, 0), 5)), tab, match="not settled")  # the winner of a tie after the draw
    _refused(bad(arg1=setv(1, [0, 1])), tab, match="taken twice")  # pair 0 twice, so pair 1 unused
    _refused(bad(arg1=setv(1, [1, 0])), tab, match="home 2i")
    _refused(bad(pairing_mode=setv(0, 7)), tab, match="mode")
    b17 = dict(good, pool_size=np.resize(good["pool_size"], 17), pairing_mode=np.resize(good["pairing_mode"], 17),
               pairing_protect=np.resize(good["pairing_protect"], 17),
               pairing_host_pot=np.resize(good["pairing_host_pot"], 17),
               **{k: np.resize(good[k], (17, 64)) for k in ("pool_kind", "pool_arg0", "pool_arg1", "pool_pot")})
    _refused(b17, tab, match="num_pairings")  # more than 16 pairings
    nogroups = season.build_table(names)
    season._size_histograms(nogroups)
    _refused(good, nogroups, match="group protection")
    # PAIRED entrants without pairings
    plain = {k: v for k, v in good.items() if k not in ("pool_kind",)}
    _refused(plain, tab, match="needs pairings")
