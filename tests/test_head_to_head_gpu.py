"""Head-to-head ranking on the GPU: the goal_difference rule through the new entry points bit-identical to the old ones,
the head_to_head kernel replayed by the float64 / integer reference (oracle/head_to_head.py) for all four models, its
positions equal to the reference ranking of its own raw scores, played matches that decide a group, draw ranges and
seeds, the 48-team World Cup through the predictor, and refusals."""
import numpy as np
import pytest

from bpl_next_b200 import _abi, problem
from oracle import head_to_head as h2h
from oracle import simulate as osim
from oracle import tournament
from tests import test_simulate_gpu as tsim
from tests import test_tournament_gpu as ttour

pytestmark = pytest.mark.gpu

MODELS = ["dixon_coles", "extended", "neutral", "neutral_wc"]


def _played(T, seed):
    """A random played head-to-head matrix [T, T, 2] (points and goals of u against v) with an empty diagonal."""
    rng = np.random.default_rng(seed)
    m = np.stack([rng.integers(0, 4, (T, T)), rng.integers(0, 3, (T, T))], axis=2).astype(np.int32)
    m[np.arange(T), np.arange(T)] = 0
    return m


def _h2h(tab, played=None):
    return dict(tab, tiebreak="head_to_head", played_h2h=played)


def _dev_table(tab):
    d = tsim._dev_table(tab)
    d.update(tiebreak=tab.get("tiebreak", "goal_difference"), played_h2h=tab.get("played_h2h"))  # (host)
    return d


def _run_table(model, s, fx, hs, as_, tab, G, R, seed, first_draw=0):
    from bpl_next_b200 import simulate_table

    out = simulate_table(model, tsim._dev(s), tsim._dev(dict(fx, home_slot=hs, away_slot=as_)), _dev_table(tab), G, R,
                         seed, first_draw=first_draw, want_positions=True, want_scores=True)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def _run_tour(model, s, fx, hs, as_, tab, br, G, R, seed, first_draw=0):
    from bpl_next_b200 import simulate_tournament

    dfx = tsim._dev(dict(fx, home_slot=hs, away_slot=as_)) if len(hs) else {}
    out = simulate_tournament(model, tsim._dev(s), dfx, _dev_table(tab), br, G, R, seed, first_draw=first_draw,
                              want_positions=True, want_scores=True, want_knockout=True)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def _forced_ranking(monkeypatch, rule, played=None):
    """Route problem._simulate through the _ex / _ranked entry points with this rule, whatever the table says."""
    def make(table, T_tab, keep):
        r = _abi.Ranking()
        r.rule = rule
        if played is not None:
            a = np.ascontiguousarray(played, np.int32)
            keep.append(a)
            r.played_h2h = a.ctypes.data
        return r

    monkeypatch.setattr(problem, "_ranking_struct", make)


def test_goal_difference_through_the_new_entry_points_is_bitwise_today(monkeypatch):
    s, fx, hs, as_, tab = tsim._case("neutral_wc", 61, 20, True, 60, seed=11)
    old = _run_table("neutral_wc", s, fx, hs, as_, tab, 15, 5, seed=7)
    s2, fx2, hs2, as2, tab2, br = ttour._case("neutral_wc", 61, 16, True, 40, seed=12, best=True)
    old_t = _run_tour("neutral_wc", s2, fx2, hs2, as2, tab2, br, 15, 5, seed=7)
    _forced_ranking(monkeypatch, _abi.RANK_GOAL_DIFF, _played(20, 1))
    new = _run_table("neutral_wc", s, fx, hs, as_, tab, 15, 5, seed=7)
    new_t = _run_tour("neutral_wc", s2, fx2, hs2, as2, tab2, br, 15, 5, seed=7)
    for a, b in ((old, new), (old_t, new_t)):
        assert set(a) == set(b)
        for k in a:
            if a[k] is not None:
                np.testing.assert_array_equal(a[k], b[k], err_msg=k)


TABLE_REPLAY = [(7, 15, 20, True, 60), (1, 15, 64, True, 100), (3, 10, 20, False, 190)]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("R,G,T_tab,grouped,F", TABLE_REPLAY)
def test_table_exact_replay(model, R, G, T_tab, grouped, F):
    """Scores equal the reference's except at rounding-level margins (as test_simulate_gpu); the kernel's positions
    equal the reference's head-to-head ranking of the kernel's own raw scores and keys, row for row (so the re-sampled
    scores of the ranking are the ones that built the table), and so do the histograms."""
    S, seed = 149, 3000 + R * 100 + T_tab
    s, fx, hs, as_, tab = tsim._case(model, S, T_tab, grouped, F, seed)
    tab = _h2h(tab, _played(T_tab, seed))
    k = _run_table(model, s, fx, hs, as_, tab, G, R, seed)
    o = h2h.simulate(model, s, fx, hs, as_, tab, G, R, seed, played_h2h=tab["played_h2h"])
    assert k["invalid"][0] == 0 and o["invalid"] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    diff = (kh != o["home"]) | (ka != o["away"])
    assert not (diff & ~(o["margin"] < 1e-5)).any()
    assert diff.sum() <= 1e-3 * diff.size
    r = h2h.rank_scores(tab, hs, as_, kh, ka, o["keys"], played_h2h=tab["played_h2h"])
    for key in ("positions", "position_counts", "points_counts"):
        np.testing.assert_array_equal(k[key], r[key], err_msg=key)
    if not diff.any():
        for key in ("positions", "position_counts", "points_counts"):
            np.testing.assert_array_equal(k[key], o[key], err_msg=key)
    # the rule changed some group orders, and only among teams level on points
    g = osim.rank_scores(tab, hs, as_, kh, ka, o["keys"])["positions"]
    pts, _, _ = osim.tables(tab, hs, as_, kh, ka)
    level = (pts[:, :, None] == pts[:, None, :]).sum(axis=2) > 1
    assert (k["positions"] != g).any() and not ((k["positions"] != g) & ~level).any()


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("R,T_tab,grouped,best,F", ttour.REPLAY)
def test_tournament_exact_replay(model, R, T_tab, grouped, best, F):
    """The group stage's scores equal the reference's except at rounding-level margins; positions are the reference's
    head-to-head ranking of the kernel's own scores; every entrant follows from those positions (best-placed
    qualifiers ranked across groups as before), the winners of earlier ties and the fixed slots; every count equals
    the counts of the kernel's own raw rows."""
    S, seed = 149, 4000 + R * 100 + T_tab + F
    s, fx, hs, as_, tab, br = ttour._case(model, S, T_tab, grouped, F, seed, best=best)
    tab = _h2h(tab, _played(T_tab, seed))
    k = _run_tour(model, s, fx, hs, as_, tab, br, 15, R, seed)
    o = tournament.simulate_tournament(model, s, fx if F else None, hs, as_, tab, br, 15, R, seed)
    assert k["invalid"][0] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    diff = (kh != o["home"]) | (ka != o["away"])
    assert not (diff & ~(o["margin"] < 1e-5)).any() and diff.sum() <= max(1, 1e-3 * diff.size)
    pos = h2h.rank(tab, hs, as_, kh, ka, o["keys"], tab["played_h2h"])
    np.testing.assert_array_equal(k["positions"], pos)
    pts, gd, gf = osim.tables(tab, hs, as_, kh, ka)
    qmap, bst, ok = tournament.qualifiers(tab, br, pts, gd, gf, o["keys"], pos)
    assert ok.all()
    ent, win = k["ko_entrants"].astype(np.int64), k["ko_winners"].astype(np.int64)
    n, K = win.shape
    for t in range(K):
        for side in range(2):
            kd, a0, a1 = (int(br[x][t, side]) for x in ("kind", "arg0", "arg1"))
            want = {_abi.ENTRANT_SLOT: lambda: np.full(n, a0), _abi.ENTRANT_GROUP_POS: lambda: qmap[:, a0, a1],
                    _abi.ENTRANT_BEST: lambda: bst[:, a0], _abi.ENTRANT_WINNER: lambda: win[:, a0],
                    _abi.ENTRANT_LOSER: lambda: ent[:, a0].sum(axis=1) - win[:, a0]}[kd]()
            np.testing.assert_array_equal(ent[:, t, side], want, err_msg=f"tie {t} side {side}")
    hist = osim.histograms(tab, pts, pos, np.ones(n, bool))
    for key in ("position_counts", "points_counts"):
        np.testing.assert_array_equal(k[key], hist[key], err_msg=key)
    T, nr = len(tab["start_points"]), int(br["num_rounds"])
    reach, wins = np.zeros((T, nr), np.int64), np.zeros((T, nr), np.int64)
    rnd = np.asarray(br["round"], np.int64)
    for t in range(K):
        np.add.at(reach, (ent[:, t, 0], rnd[t]), 1)
        np.add.at(reach, (ent[:, t, 1], rnd[t]), 1)
        np.add.at(wins, (win[:, t], rnd[t]), 1)
    np.testing.assert_array_equal(k["reach_counts"], reach)
    np.testing.assert_array_equal(k["win_counts"], wins)
    # the knockout ties between the same entrants are played as under goal_difference: the same words, the same code
    g = _run_tour(model, s, fx, hs, as_, dict(tab, tiebreak="goal_difference"), br, 15, R, seed)
    same = (g["ko_entrants"] == k["ko_entrants"]).all(axis=(1, 2))
    assert same.any()
    for key in ("ko_scores", "ko_winners", "scores"):
        np.testing.assert_array_equal(g[key][same], k[key][same], err_msg=key)


def test_played_matches_decide():
    """One group of four level at the start, and a played round in which slot 0 beat every other team 1-0: the
    kernel's positions are the reference's ranking with those played matches, the same simulations without them are
    ranked as the reference ranks them without, and the played matches change some orders."""
    s, fx, hs, as_, tab = tsim._case("dixon_coles", 200, 4, False, 6 * 2, seed=21)
    for k in ("start_points", "start_goals_for", "start_goals_against"):
        tab[k] = np.zeros(4, np.int32)
    played = np.zeros((4, 4, 2), np.int32)
    played[0, 1:] = (3, 1)
    with_p = _run_table("dixon_coles", s, fx, hs, as_, _h2h(tab, played), 15, 8, seed=5)
    without = _run_table("dixon_coles", s, fx, hs, as_, _h2h(tab), 15, 8, seed=5)
    np.testing.assert_array_equal(with_p["scores"], without["scores"])
    kh, ka = with_p["scores"][:, :, 0].astype(np.int64), with_p["scores"][:, :, 1].astype(np.int64)
    keys = osim.philox_words(s, 8, 5, 0, 2 * len(hs) + 4)[0][:, 2 * len(hs):].astype(np.int64)
    np.testing.assert_array_equal(with_p["positions"], h2h.rank(tab, hs, as_, kh, ka, keys, played))
    np.testing.assert_array_equal(without["positions"], h2h.rank(tab, hs, as_, kh, ka, keys))
    assert (with_p["positions"] != without["positions"]).any()


def test_draw_ranges_and_seeds():
    s, fx, hs, as_, tab = tsim._case("neutral_wc", 50, 12, True, 40, seed=5)
    tab = _h2h(tab, _played(12, 3))
    full = _run_table("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=99)
    parts = [_run_table("neutral_wc", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, 15, 3, seed=99,
                       first_draw=lo) for lo, hi in ((0, 17), (17, 50))]
    for key in ("position_counts", "points_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key])
    for key in ("positions", "scores"):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]))
    again = _run_table("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=99)
    for key in ("position_counts", "points_counts", "positions", "scores"):
        np.testing.assert_array_equal(full[key], again[key])
    other = _run_table("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=100)
    assert not np.array_equal(full["scores"], other["scores"])
    s2, fx2, hs2, as2, tab2, br = ttour._case("neutral", 40, 16, True, 40, seed=6, best=True)
    tab2 = _h2h(tab2)
    full = _run_tour("neutral", s2, fx2, hs2, as2, tab2, br, 15, 4, seed=3)
    parts = [_run_tour("neutral", {k: v[lo:hi] for k, v in s2.items()}, fx2, hs2, as2, tab2, br, 15, 4, seed=3,
                        first_draw=lo) for lo, hi in ((0, 13), (13, 40))]
    for key in ("position_counts", "points_counts", "reach_counts", "win_counts", "decided_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key], err_msg=key)
    for key in ("positions", "ko_entrants", "ko_winners"):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]), err_msg=key)


def test_world_cup_48_end_to_end():
    """The 48-team World Cup through the predictor under both rules with one seed: the same scores and points; group
    orders differ only among teams level on points; the best thirds and every entrant follow from the head-to-head
    positions by the unchanged cross-group ranking."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor

    m = ttour._wc_predictor(S=128)
    teams, groups, fx, ties, best = ttour._world_cup_48()
    kw = dict(groups=groups, best=best, num_sims_per_draw=4, random_state=17, return_simulations=True)
    gd = m.simulate_tournament(fx, ties, **kw)
    hh = m.simulate_tournament(fx, ties, tiebreak="head_to_head", **kw)
    assert gd["tiebreak"] == "goal_difference" and hh["tiebreak"] == "head_to_head"
    for key in ("home_score", "away_score", "points_proba", "expected_points"):
        np.testing.assert_array_equal(gd[key], hh[key], err_msg=key)
    assert not np.array_equal(gd["position_proba"], hh["position_proba"])
    np.testing.assert_allclose(hh["champion_proba"].sum(), 1.0, rtol=0, atol=1e-12)
    # the reference's ranking of the kernel's own scores, and the qualifiers it implies
    from bpl_next_b200 import season

    tab = season.build_table(teams, groups=groups, tiebreak="head_to_head")
    hs, as_ = season.fixture_slots(tab, fx["home_team"], fx["away_team"])
    br = season.build_bracket(tab, ties, best)
    kh, ka = hh["home_score"].T.astype(np.int64), hh["away_score"].T.astype(np.int64)
    F, N = len(hs), kh.shape[0]
    keys = osim.philox_words({"attack": m.attack}, 4, 17, 0, 2 * F + 48)[0][:, 2 * F:].astype(np.int64)
    pts, gdv, gf = osim.tables(tab, hs, as_, kh, ka)
    level = (pts[:, :, None] == pts[:, None, :]).sum(axis=2) > 1
    assert not ((hh["positions"] != gd["positions"]) & ~level).any()
    np.testing.assert_array_equal(hh["positions"], h2h.rank(tab, hs, as_, kh, ka, keys))
    qmap, _, _ = tournament.qualifiers(tab, br, pts, gdv, gf, np.zeros((N, 48), np.int64), hh["positions"])
    thirds = qmap[:, :, 2]  # [N, 12]
    ent = hh["ko_entrants"].astype(np.int64)
    kind = np.asarray(br["kind"])
    # the eight best thirds: no third outside them ranks above one of them across groups
    best_slots = np.stack([ent[:, t, s] for t in range(len(ties)) for s in range(2)
                           if kind[t, s] == _abi.ENTRANT_BEST], axis=1)
    assert best_slots.shape == (N, 8)
    for i in range(N):
        chosen = set(best_slots[i].tolist())
        assert chosen <= set(thirds[i].tolist())
        worst = min((pts[i, t], gdv[i, t], gf[i, t]) for t in chosen)
        assert all((pts[i, t], gdv[i, t], gf[i, t]) <= worst for t in set(thirds[i].tolist()) - chosen)
    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().simulate_tournament(fx, ties, tiebreak="head_to_head")


def test_refusals(monkeypatch):
    s, fx, hs, as_, tab = tsim._case("dixon_coles", 8, 8, False, 20, seed=31)
    with pytest.raises(ValueError, match="unknown tiebreak"):
        _run_table("dixon_coles", s, fx, hs, as_, dict(tab, tiebreak="fair_play"), 15, 2, seed=1)
    bad = _played(8, 2)
    bad[1, 2, 1] = -1
    with pytest.raises(_abi.BplxError, match="negative"):
        _run_table("dixon_coles", s, fx, hs, as_, _h2h(tab, bad), 15, 2, seed=1)
    s2, fx2, hs2, as2, tab2, br = ttour._case("dixon_coles", 8, 8, False, 20, seed=32)
    with pytest.raises(_abi.BplxError, match="negative"):
        _run_tour("dixon_coles", s2, fx2, hs2, as2, _h2h(tab2, bad), br, 15, 2, seed=1)
    _forced_ranking(monkeypatch, 7)
    with pytest.raises(_abi.BplxError, match="ranking rule 7"):
        _run_table("dixon_coles", s, fx, hs, as_, tab, 15, 2, seed=1)
    with pytest.raises(_abi.BplxError, match="ranking rule 7"):
        _run_tour("dixon_coles", s2, fx2, hs2, as2, tab2, br, 15, 2, seed=1)
    with pytest.raises(_abi.BplxError):
        _run_table("dynamic", s, fx, hs, as_, _h2h(tab), 15, 2, seed=1)
