"""Head-to-head ranking on the CPU: hand-worked groups through the integer reference under both rules,
``season.build_table``'s played head-to-head matrix and refusals, and the ctypes struct and prototypes against the
header."""
import ctypes as C
import re

import numpy as np
import pytest

from bpl_next_b200 import _abi, problem, season
from oracle import head_to_head as h2h
from oracle import simulate as osim

TEAMS = ["A", "B", "C", "D"]


def _positions(results, played=None, tiebreak="head_to_head", keys=(0, 0, 0, 0)):
    """The order (team names, first to last) of one group: ``results`` are the simulated fixtures as
    ``(home, away, home goals, away goals)``, ``played`` the played ones."""
    pl = None
    if played:
        pl = {"home_team": [r[0] for r in played], "away_team": [r[1] for r in played],
              "home_goals": [r[2] for r in played], "away_goals": [r[3] for r in played]}
    tab = season.build_table(TEAMS, pl, tiebreak=tiebreak)
    hs, as_ = season.fixture_slots(tab, [r[0] for r in results], [r[1] for r in results])
    home = np.asarray([[r[2] for r in results]])
    away = np.asarray([[r[3] for r in results]])
    pos = h2h.rank(tab, hs, as_, home, away, np.asarray([keys]), tab.get("played_h2h"), tiebreak)[0]
    return "".join(TEAMS[t] for t in np.argsort(pos))


# the three hand-worked groups: results, goal_difference order, head_to_head order
HAND = [
    # two teams level on points: head-to-head beats a better goal difference
    ([("A", "B", 1, 0), ("A", "D", 1, 0), ("C", "A", 1, 0), ("B", "C", 3, 0), ("B", "D", 3, 0), ("C", "D", 0, 0)],
     "BACD", "ABCD"),
    # three-way circle: C is separated on head-to-head goals for, then A-B is reapplied to their own match
    ([("A", "B", 1, 0), ("A", "C", 1, 2), ("B", "C", 2, 1), ("A", "D", 1, 0), ("B", "D", 5, 0), ("C", "D", 1, 0)],
     "BCAD", "CABD"),
    # head-to-head separates nobody, so overall goal difference decides
    ([("A", "B", 1, 1), ("A", "C", 1, 1), ("B", "C", 1, 1), ("A", "D", 1, 0), ("B", "D", 3, 0), ("C", "D", 2, 0)],
     "BCAD", "BCAD"),
]


@pytest.mark.parametrize("results,gd_order,h2h_order", HAND)
def test_hand_worked_groups(results, gd_order, h2h_order):
    assert _positions(results, tiebreak="goal_difference") == gd_order
    assert _positions(results, tiebreak="head_to_head") == h2h_order


def test_three_way_circle_is_reapplied_not_sent_to_goal_difference():
    results = HAND[1][0]
    tab = season.build_table(TEAMS, tiebreak="head_to_head")
    hs, as_ = season.fixture_slots(tab, [r[0] for r in results], [r[1] for r in results])
    pair = h2h.pair_results(tab, hs, as_, [r[2] for r in results], [r[3] for r in results])
    # A, B, C are level on 6 points; among them C scored 3, A and B 2 each, with the same points and goal difference
    pts, gd, gf = osim.tables(tab, hs, as_, np.asarray([[r[2] for r in results]]), np.asarray([[r[3] for r in results]]))
    assert list(pts[0, :3]) == [6, 6, 6]
    assert h2h.order_level_set([0, 1, 2], pair, gd[0], gf[0], np.zeros(4)) == [2, 0, 1]
    # falling straight to overall goal difference after C would put B before A
    assert sorted([0, 1], key=lambda x: (-gd[0, x], -gf[0, x])) == [1, 0]


def test_teams_that_have_not_met_fall_through_to_goal_difference():
    # A and B level on 3 points without a match between them: B's better goal difference decides; C and D drew
    results = [("A", "C", 1, 0), ("B", "D", 2, 0), ("C", "D", 0, 0)]
    assert _positions(results, tiebreak="head_to_head") == "BACD"
    assert _positions(results, tiebreak="goal_difference") == "BACD"
    # fully level (points, goal difference, goals for, no match between them): the key, then the lower slot
    results = [("A", "C", 1, 0), ("B", "D", 1, 0)]
    assert _positions(results, keys=(1, 5, 0, 0))[:2] == "BA"
    assert _positions(results, keys=(7, 7, 0, 0))[:2] == "AB"


def test_only_a_played_match_separates_two_teams():
    # A beat B in a played match; the rest of the season leaves them level on 4 points with B ahead on goal difference
    played = [("A", "B", 1, 0)]
    results = [("A", "C", 0, 0), ("B", "C", 4, 0), ("B", "D", 0, 0)]
    assert _positions(results, played, tiebreak="goal_difference") == "BADC"
    assert _positions(results, played, tiebreak="head_to_head") == "ABDC"


def test_goal_difference_rule_is_todays_rank():
    rng = np.random.default_rng(3)
    T, F, n = 8, 20, 400
    tab = season.build_table([f"t{k}" for k in range(T)], groups=[k % 2 for k in range(T)])
    hs = rng.integers(0, T, F)
    as_ = (hs + 2 * rng.integers(1, T // 2, F)) % T  # the same group
    home, away = rng.integers(0, 3, (n, F)), rng.integers(0, 3, (n, F))
    keys = rng.integers(0, 2 ** 32, (n, T))
    pts, gd, gf = osim.tables(tab, hs, as_, home, away)
    np.testing.assert_array_equal(h2h.rank(tab, hs, as_, home, away, keys, tiebreak="goal_difference"),
                                  osim.rank(pts, gd, gf, keys, tab["group"]))
    # head-to-head only reorders teams level on points
    pos = h2h.rank(tab, hs, as_, home, away, keys)
    gpos = osim.rank(pts, gd, gf, keys, tab["group"])
    level = (pts[:, :, None] == pts[:, None, :]).sum(axis=2) > 1  # a team level on points with another
    grp = tab["group"]
    for i in range(n):
        for g in (0, 1):
            mem = np.flatnonzero(grp == g)
            assert sorted(pos[i, mem]) == list(range(len(mem)))
            order = mem[np.argsort(pos[i, mem])]
            assert (np.diff(pts[i, order]) <= 0).all()
    assert ((pos != gpos) <= level).all()
    assert (pos != gpos).any()


def test_build_table_played_matrix_and_refusals():
    played = {"home_team": ["A", "B", "C"], "away_team": ["B", "A", "D"], "home_goals": [2, 1, 0],
              "away_goals": [0, 1, 3]}
    gd = season.build_table(TEAMS, played)
    assert gd["tiebreak"] == "goal_difference" and "played_h2h" not in gd
    tab = season.build_table(TEAMS, played, points=(3, 1), tiebreak="head_to_head")
    m = tab["played_h2h"]
    assert m.dtype == np.int32 and m.shape == (4, 4, 2)
    assert tuple(m[0, 1]) == (4, 3) and tuple(m[1, 0]) == (1, 1)  # A: a win and a draw against B, 2 + 1 goals
    assert tuple(m[2, 3]) == (0, 0) and tuple(m[3, 2]) == (3, 3)
    assert m[[0, 1, 2, 3], [0, 1, 2, 3]].sum() == 0 and m[0, 2:].sum() == 0
    for k in ("start_points", "start_goals_for", "start_goals_against"):
        np.testing.assert_array_equal(tab[k], gd[k])
    with pytest.raises(ValueError, match="unknown tiebreak"):
        season.build_table(TEAMS, played, tiebreak="fair_play")
    with pytest.raises(ValueError, match="unknown tiebreak"):
        problem._ranking_struct({"tiebreak": "away_goals"}, 4, [])
    with pytest.raises(ValueError, match="played_h2h has shape"):
        problem._ranking_struct({"tiebreak": "head_to_head", "played_h2h": np.zeros((3, 3, 2))}, 4, [])
    assert problem._ranking_struct(gd, 4, []) is None
    assert season.TIEBREAKS == {"goal_difference": _abi.RANK_GOAL_DIFF, "head_to_head": _abi.RANK_HEAD_TO_HEAD}


def _params(text, name):
    proto = re.search(r"\b" + name + r"\(([^;]*)\);", text).group(1)
    return [re.split(r"[ *]+", p.strip())[-1] for p in proto.split(",")]


def test_struct_and_prototypes_match_the_header():
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    assert "#define BPLX_RANK_GOAL_DIFF 0" in text and "#define BPLX_RANK_HEAD_TO_HEAD 1" in text
    assert (_abi.RANK_GOAL_DIFF, _abi.RANK_HEAD_TO_HEAD) == (0, 1)
    assert "#define BPLX_VERSION 1" in text
    body = re.search(r"typedef struct \{([^}]*)\} bplx_ranking;", text).group(1)
    assert re.findall(r"^\s*(.*?)\s*(\w+);", body, re.M) == [("int32_t", "rule"), ("const int32_t*", "played_h2h")]
    assert [f[0] for f in _abi.Ranking._fields_] == ["rule", "played_h2h"]
    assert C.sizeof(_abi.Ranking) == 16 and _abi.Ranking.played_h2h.offset == 8
    lib = _abi.lib()
    # the table call with the ranking after the table; the tournament call with it after tie_format
    table, ex = _params(text, "bplx_simulate_table"), _params(text, "bplx_simulate_table_ex")
    assert [n for n in ex if n != "r"] == table and ex.index("r") == ex.index("t") + 1
    assert len(lib.bplx_simulate_table_ex.argtypes) == len(ex) == 18
    tour, ranked = _params(text, "bplx_simulate_tournament_ex"), _params(text, "bplx_simulate_tournament_ranked")
    assert [n for n in ranked if n != "r"] == tour and ranked.index("r") == ranked.index("tie_format") + 1
    assert len(lib.bplx_simulate_tournament_ranked.argtypes) == len(ranked) == 27
    for fn, n in (("bplx_simulate_table_ex_workspace_bytes", 4), ("bplx_simulate_tournament_ranked_workspace_bytes", 5)):
        params = _params(text, fn)
        assert len(getattr(lib, fn).argtypes) == len(params) == n and params[-1] == "r"
        assert getattr(lib, fn).restype == C.c_size_t
    for fn in ("bplx_simulate_table_ex", "bplx_simulate_tournament_ranked"):
        assert getattr(lib, fn).restype == C.c_int
        ri = _params(text, fn).index("r")
        assert getattr(lib, fn).argtypes[ri] == C.POINTER(_abi.Ranking)
