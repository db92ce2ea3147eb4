"""Tournament simulation on the CPU: bracket validation in ``season.build_bracket``, the best-placed ranking and the
allocation lookup of the float64 oracle on hand-built tables, the oracle's decider against the exact per-draw
``hw / (hw + aw)``, ``resolve_bracket`` on hand-written scores, and the ctypes ``Bracket`` against the header."""
import ctypes as C
import itertools

import numpy as np
import pytest

from bpl_next_b200 import _abi, season
from oracle import philox
from oracle import simulate as osim
from oracle import tournament


def _groups(n_groups, size=4):
    teams = [f"{chr(65 + g)}{i}" for g in range(n_groups) for i in range(size)]
    return teams, {t: t[0] for t in teams}


def _alloc(labels, count):
    """A complete allocation: every count-subset of the groups, BEST j = the subset's groups rotated by its size."""
    out = {}
    for sub in itertools.combinations(labels, count):
        r = len(out) % count
        out[frozenset(sub)] = list(sub[r:] + sub[:r])
    return out


def _euro():
    """24 teams in 6 groups of four; R16 of winners, runners-up and the 4 best thirds, then QF, SF, final."""
    teams, groups = _groups(6)
    tab = season.build_table(teams, groups=groups)
    L = list("ABCDEF")
    r16 = []
    for k in range(6):
        away = ("best", k) if k < 4 else ("group", L[(k + 1) % 6], 1)
        r16.append({"id": f"r{k}", "round": "R16", "home": ("group", L[k], 0), "away": away})
    r16 += [{"id": "r6", "round": "R16", "home": ("group", "B", 1), "away": ("group", "C", 1)},
            {"id": "r7", "round": "R16", "home": ("group", "D", 1), "away": ("group", "E", 1)}]
    qf = [{"id": f"q{k}", "round": "QF", "home": ("winner", f"r{2 * k}"), "away": ("winner", f"r{2 * k + 1}")}
          for k in range(4)]
    sf = [{"id": f"s{k}", "round": "SF", "home": ("winner", f"q{2 * k}"), "away": ("winner", f"q{2 * k + 1}")}
          for k in range(2)]
    final = [{"id": "f", "round": "F", "home": ("winner", "s0"), "away": ("winner", "s1"), "neutral_venue": 1}]
    return tab, r16 + qf + sf + final


def test_build_bracket_euro_layout():
    tab, ties = _euro()
    best = {"position": 2, "count": 4, "allocation": _alloc(list("ABCDEF"), 4)}
    b = season.build_bracket(tab, ties, best)
    assert b["rounds"] == ["R16", "QF", "SF", "F"] and b["num_rounds"] == 4 and b["num_groups"] == 6
    assert b["best_alloc"].shape == (64, 4)
    assert (b["best_alloc"] != 255).all(axis=1).sum() == 15  # the 15 four-of-six rows, the rest 0xFF
    np.testing.assert_array_equal(b["kind"][0], [season.ENTRANT_GROUP_POS, season.ENTRANT_BEST])
    np.testing.assert_array_equal(b["kind"][8], [season.ENTRANT_WINNER, season.ENTRANT_WINNER])
    np.testing.assert_array_equal(b["arg0"][8], [0, 1])
    assert b["neutral_venue"][-1] == 1 and b["neutral_venue"][0] == 0


def test_build_bracket_refusals():
    tab, ties = _euro()
    best = {"position": 2, "count": 4}
    with pytest.raises(ValueError, match="used twice"):
        bad = [dict(t) for t in ties]
        bad[1]["home"] = ("group", "A", 0)
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="used twice"):
        bad = [dict(t) for t in ties]
        bad[9]["away"] = ("winner", "q0")
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="unknown tie id"):
        bad = [dict(t) for t in ties]
        bad[8]["home"] = ("winner", "nope")
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="not played before it"):
        bad = [dict(t) for t in ties]
        bad[8]["home"] = ("winner", "q3")
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="used twice"):
        bad = [dict(t) for t in ties]
        bad[1]["id"] = "r0"
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="not one of the 4 best"):
        bad = [dict(t) for t in ties]
        bad[0]["away"] = ("best", 4)
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="no position 4"):
        bad = [dict(t) for t in ties]
        bad[0]["home"] = ("group", "A", 4)
        season.build_bracket(tab, bad, best)
    with pytest.raises(ValueError, match="alone in its round"):
        season.build_bracket(tab, ties[:-1], best)
    al = _alloc(list("ABCDEF"), 4)
    missing = dict(al)
    missing.pop(frozenset("ABCD"))
    with pytest.raises(ValueError, match="misses"):
        season.build_bracket(tab, ties, dict(best, allocation=missing))
    notperm = dict(al)
    notperm[frozenset("ABCD")] = ["A", "B", "C", "E"]
    with pytest.raises(ValueError, match="permutation"):
        season.build_bracket(tab, ties, dict(best, allocation=notperm))
    with pytest.raises(ValueError, match="1 to 64 ties"):
        season.build_bracket(tab, [], best)


def _euro_case(seed):
    """Hand-built final group tables of the Euro layout (integers) with positions from the oracle's ranking."""
    rng = np.random.default_rng(seed)
    tab, ties = _euro()
    best = {"position": 2, "count": 4, "allocation": _alloc(list("ABCDEF"), 4)}
    b = season.build_bracket(tab, ties, best)
    n, T = 200, 24
    pts = rng.integers(0, 4, (n, T))  # few distinct values: many level thirds
    gd = rng.integers(-1, 2, (n, T))
    gf = rng.integers(0, 2, (n, T))
    keys = rng.integers(0, 2 ** 32, (n, T))
    keys[:, 5] = keys[:, 9]  # some keys equal: the lower slot decides
    pos = osim.rank(pts, gd, gf, keys, tab["group"])
    return tab, b, pts, gd, gf, keys, pos


def test_best_placed_ranking_and_allocation_lookup():
    """Six groups of four, the four best thirds: the oracle's pool ranking by brute force over the thirds, and BEST j
    = the third of group alloc[mask][j] with the generated 15-row table."""
    tab, b, pts, gd, gf, keys, pos = _euro_case(1)
    qmap, best, ok = tournament.qualifiers(tab, b, pts, gd, gf, keys, pos)
    assert ok.all()
    group = tab["group"].astype(np.int64)
    for i in range(pts.shape[0]):
        thirds = [int(np.flatnonzero((group == g) & (pos[i] == 2))[0]) for g in range(6)]
        order = sorted(thirds, key=lambda t: (-pts[i, t], -gd[i, t], -gf[i, t], -keys[i, t], t))
        top = order[:4]
        mask = sum(1 << int(group[t]) for t in top)
        row = b["best_alloc"][mask]
        assert sorted(row.tolist()) == sorted(int(group[t]) for t in top)
        np.testing.assert_array_equal(best[i], [thirds[g] for g in row])
        for g in range(6):
            for p in range(4):
                assert pos[i, qmap[i, g, p]] == p and group[qmap[i, g, p]] == g
    # without an allocation, BEST j is the j-th best third
    nb = dict(b, best_alloc=None)
    _, best2, ok2 = tournament.qualifiers(tab, nb, pts, gd, gf, keys, pos)
    i = 0
    thirds = [int(np.flatnonzero((group == g) & (pos[i] == 2))[0]) for g in range(6)]
    order = sorted(thirds, key=lambda t: (-pts[i, t], -gd[i, t], -gf[i, t], -keys[i, t], t))
    np.testing.assert_array_equal(best2[0], order[:4])
    # an allocation row of 0xFF makes the simulation invalid
    bad = dict(b, best_alloc=b["best_alloc"].copy())
    bad["best_alloc"][:] = 255
    assert not tournament.qualifiers(tab, bad, pts, gd, gf, keys, pos)[2].any()


@pytest.mark.parametrize("lh,la,c", [(1.6, 1.1, -0.12), (0.4, 2.7, 0.3), (1.0, 1.0, 0.0), (0.2, 0.3, 5.0)])
def test_decider_against_the_exact_per_draw_ratio(lh, la, c):
    """N = 2e5 drawn ties of one draw: the share the oracle gives the home entrant is within 5 sigma of hw / (hw + aw)
    computed on the full clamped grid, and its win masses equal that grid's (off-diagonal sums)."""
    from oracle import predict as op

    G = 15
    hw, aw = tournament.win_masses(np.array([lh]), np.array([la]), np.array([c]), G)
    samples = {"attack": np.array([[np.log(lh), np.log(la)]]), "defence": np.zeros((1, 2)),
               "home_advantage": np.zeros(1), "corr_coef": np.array([c])}
    grid, _, _ = op.predict_score_grid_proba("dixon_coles", samples, [0], [1], G)
    g = np.maximum(grid[0], 0.0)
    ehw, eaw = np.tril(g, -1).sum(), np.triu(g, 1).sum()
    np.testing.assert_allclose(hw[0] / (hw[0] + aw[0]), ehw / (ehw + eaw), rtol=1e-12)
    N = 200_000
    u = philox.uniform(philox.stream(3, np.arange(N, dtype=np.uint64), 0, 1)[:, 0]).astype(np.float64)
    p = hw[0] / (hw[0] + aw[0])
    share = (u * (hw[0] + aw[0]) <= hw[0]).mean()
    assert abs(share - p) <= 5 * np.sqrt(p * (1 - p) / N) + 1e-12


def test_resolve_bracket_by_hand():
    """Two groups of three, the winners and runners-up cross over, the best third (one of two) plays a fixed team in
    a play-in, then the final and a third-place match; every entrant, winner and count by hand."""
    teams = ["A0", "A1", "A2", "B0", "B1", "B2", "X"]
    groups = {"A0": "A", "A1": "A", "A2": "A", "B0": "B", "B1": "B", "B2": "B", "X": "Z"}
    tab = season.build_table(teams, groups=groups)
    pairs = [("A0", "A1"), ("A0", "A2"), ("A1", "A2"), ("B0", "B1"), ("B0", "B2"), ("B1", "B2")]
    hs, as_ = season.fixture_slots(tab, [p[0] for p in pairs], [p[1] for p in pairs])
    ties = [{"id": "p", "round": "play-in", "home": ("team", "X"), "away": ("best", 0)},
            {"id": "s1", "round": "SF", "home": ("group", "A", 0), "away": ("group", "B", 1)},
            {"id": "s2", "round": "SF", "home": ("group", "B", 0), "away": ("winner", "p")},
            {"id": "3rd", "round": "third", "home": ("loser", "s1"), "away": ("loser", "s2")},
            {"id": "f", "round": "F", "home": ("winner", "s1"), "away": ("winner", "s2")}]
    b = season.build_bracket(tab, ties, {"position": 2, "count": 1})
    assert b["rounds"] == ["play-in", "SF", "third", "F"]
    # group A: A0 beats both, A1 beats A2 -> A0, A1, A2 (A2: 0 pts, gd -3); group B: all 1-1 draws, keys decide
    home = np.array([[2, 1, 1, 1, 1, 1]])
    away = np.array([[0, 0, 0, 1, 1, 1]])
    keys = np.array([[0, 0, 0, 5, 9, 7, 0]])  # B1 > B2 > B0 on the key; B0 is third with 2 pts beats A2's 0
    # ties: play-in X-B0 1-1, home through; s1 A0-B2 0-2; s2 B1-X 3-0; third A0-B1 2-2 away through; final B2-B1 0-1
    ko_h = np.array([[1, 0, 3, 2, 0]])
    ko_a = np.array([[1, 2, 0, 2, 1]])
    through = np.array([[1, 0, 0, 0, 0]])
    r = tournament.resolve_bracket(dict(tab, num_positions=3, num_points_bins=7), hs, as_, b, home, away, keys, ko_h,
                                   ko_a, through)
    slot = {t: i for i, t in enumerate(teams)}
    e = [[slot[x] for x in pair] for pair in (("X", "B0"), ("A0", "B2"), ("B1", "X"), ("A0", "X"), ("B2", "B1"))]
    np.testing.assert_array_equal(r["ko_entrants"][0], e)
    np.testing.assert_array_equal(r["ko_winners"][0], [slot[t] for t in ("X", "B2", "B1", "X", "B1")])
    assert r["valid"].all() and r["invalid"] == 0
    reach, win = r["reach_counts"], r["win_counts"]
    assert reach[slot["X"]].tolist() == [1, 1, 1, 0] and win[slot["X"]].tolist() == [1, 0, 1, 0]
    assert reach[slot["B1"]].tolist() == [0, 1, 0, 1] and win[slot["B1"]].tolist() == [0, 1, 0, 1]
    assert reach.sum(axis=0).tolist() == [2, 4, 2, 2] and win.sum(axis=0).tolist() == [1, 2, 1, 1]
    np.testing.assert_array_equal(r["positions"][0], [0, 1, 2, 2, 0, 1, 0])
    pr = season.bracket_probabilities(b, reach, win, 1)
    assert pr["champion_proba"][slot["B1"]] == 1.0 and pr["champion_proba"].sum() == 1.0


def test_bracket_struct_matches_header():
    assert C.sizeof(_abi.Bracket) == 5 * 4 + 4 + 8 * 8  # 5 int32, padding, 8 pointers
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    for name, val in (("BPLX_KO_MAX_TIES", _abi.KO_MAX_TIES), ("BPLX_KO_MAX_ROUNDS", _abi.KO_MAX_ROUNDS),
                      ("BPLX_KO_MAX_BEST", _abi.KO_MAX_BEST), ("BPLX_ENTRANT_LOSER", _abi.ENTRANT_LOSER),
                      ("BPLX_ENTRANT_GROUP_POS", _abi.ENTRANT_GROUP_POS)):
        assert f"#define {name} {val}" in text
