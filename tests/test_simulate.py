"""Season / group-stage simulation on the CPU: the float64 oracle's score sampler against the exact per-draw grid, its
ranking on hand-built tables, and the host arithmetic of ``bpl_next_b200.season`` (starting table, slots, validation)."""
import numpy as np
import pytest

from bpl_next_b200 import season
from oracle import philox
from oracle import predict as op
from oracle import simulate as osim


@pytest.mark.parametrize("max_goals", [15, 4])
@pytest.mark.parametrize("lh,la,c", [(1.6, 1.1, -0.12), (0.4, 2.7, 0.3), (3.5, 0.2, 5.0)])
def test_sampler_frequencies_match_the_grid(max_goals, lh, la, c):
    """N = 2e5 simulations of one draw: every cell's count is within 5 sigma (+1) of N times the draw's grid from
    oracle/predict.py (tau clamped at 0), normalised by its sum; cells of probability 0 are never drawn."""
    N = 200_000
    words = philox.stream(7, np.arange(N, dtype=np.uint64), 0, 2)
    u = philox.uniform(words).astype(np.float64)
    ones = np.ones(N)
    hg, ag, margin, valid = osim.sample_scores(lh * ones, la * ones, c * ones, u[:, 0], u[:, 1], max_goals)
    assert valid.all() and (margin >= 0).all()
    samples = {"attack": np.array([[np.log(lh), np.log(la)]]), "defence": np.zeros((1, 2)),
               "home_advantage": np.zeros(1), "corr_coef": np.array([c])}
    grid, _, _ = op.predict_score_grid_proba("dixon_coles", samples, [0], [1], max_goals)
    p = grid[0] / grid[0].sum()
    g = max_goals + 1
    counts = np.bincount(hg * g + ag, minlength=g * g).reshape(g, g)
    exp = N * p
    assert (np.abs(counts - exp) <= 5 * np.sqrt(exp * (1 - p)) + 1).all()
    assert (counts[p == 0] == 0).all()
    if c == 5.0:
        assert counts[0, 0] == 0 and counts[1, 1] == 0


def test_ranking_criteria_in_order():
    """Points > goal difference > goals for > tie-break key > lower slot, all descending but the slot."""
    # slots:        0   1   2   3   4   5
    pts = np.array([[10, 12, 10, 10, 10, 10]])
    gd = np.array([[5, -3, 5, 5, 7, 5]])
    gf = np.array([[9, 1, 9, 11, 2, 9]])
    key = np.array([[4, 0, 4, 0, 0, 9]])
    # 1 (12 pts); 4 (10, gd 7); 3 (gf 11); 5 (key 9); 0 and 2 tie on everything: the lower slot first
    np.testing.assert_array_equal(osim.rank(pts, gd, gf, key), [[4, 0, 5, 2, 1, 3]])
    # groups: each group ranked on its own
    group = np.array([0, 0, 0, 1, 1, 1])
    np.testing.assert_array_equal(osim.rank(pts, gd, gf, key, group), [[1, 0, 2, 1, 0, 2]])


def test_tables_and_histograms_from_scores():
    """Three fixtures of a four-team table, with a start from `played`; positions and gained points by hand."""
    played = {"home_team": ["A", "C"], "away_team": ["B", "D"], "home_goals": [2, 1], "away_goals": [0, 1]}
    tab = season.build_table(["A", "B", "C", "D"], played)
    np.testing.assert_array_equal(tab["start_points"], [3, 0, 1, 1])
    np.testing.assert_array_equal(tab["start_goals_for"], [2, 0, 1, 1])
    np.testing.assert_array_equal(tab["start_goals_against"], [0, 2, 1, 1])
    hs, as_ = season.fixture_slots(tab, ["B", "D", "A"], ["C", "A", "C"])
    assert tab["num_positions"] == 4 and tab["num_points_bins"] == 3 * 2 + 1
    home = np.array([[1, 3, 0], [0, 0, 0]])
    away = np.array([[0, 3, 2], [0, 0, 0]])
    out = osim.rank_scores(tab, hs, as_, home, away, keys=np.zeros((2, 4), np.int64))
    # sim 0: B beats C (B 3 pts), D-A 3-3 (A 4, D 2), A loses 0-2 to C (C 4): A 4 pts gd 2-0+3-3+0-2 = 0, gf 5;
    #        C 4 pts gd 0 + (-1) + 2 = 1 -> C first, A second, B 3 pts third, D 2 pts fourth
    np.testing.assert_array_equal(out["positions"][0], [1, 2, 0, 3])
    # sim 1: three 0-0 draws: A 5 (gd 2), C 3 (gd 0, gf 1), D 2, B 1
    np.testing.assert_array_equal(out["positions"][1], [0, 3, 1, 2])
    np.testing.assert_array_equal(out["points_counts"][:, :4], [[0, 1, 1, 0], [0, 1, 0, 1], [0, 0, 1, 1], [0, 2, 0, 0]])
    np.testing.assert_array_equal(out["position_counts"].sum(axis=0), [2, 2, 2, 2])


def test_oracle_simulation_is_a_function_of_the_draw_ranges():
    """Draws [0, 3) and [3, 5) with first_draw give the rows and counts of the single run; a different seed differs."""
    rng = np.random.default_rng(3)
    S, T = 5, 4
    s = {"attack": rng.normal(0, 0.3, (S, T)), "defence": rng.normal(0, 0.3, (S, T)),
         "home_advantage": rng.normal(0.2, 0.05, S), "corr_coef": rng.uniform(-0.1, 0.1, S)}
    tab = season.build_table(list("ABCD"))
    home, away = ["A", "B", "C", "D", "A", "C"], ["B", "C", "D", "A", "C", "B"]
    hs, as_ = season.fixture_slots(tab, home, away)
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16)}
    full = osim.simulate("dixon_coles", s, fx, hs, as_, tab, 15, 3, seed=11)
    parts = [osim.simulate("dixon_coles", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, 15, 3, seed=11,
                           first_draw=lo) for lo, hi in ((0, 3), (3, 5))]
    for k in ("home", "away", "positions"):
        np.testing.assert_array_equal(full[k], np.concatenate([p[k] for p in parts]))
    for k in ("position_counts", "points_counts"):
        np.testing.assert_array_equal(full[k], parts[0][k] + parts[1][k])
    other = osim.simulate("dixon_coles", s, fx, hs, as_, tab, 15, 3, seed=12)
    assert not np.array_equal(full["home"], other["home"])
    assert full["invalid"] == 0 and full["position_counts"].sum() == 15 * T


def test_season_validation():
    tab = season.build_table(["A", "B", "C"])
    with pytest.raises(ValueError, match="not known to the model"):
        season.fixture_slots(tab, ["A"], ["Z"], known_teams=["A", "B", "C", "Z0"])
    with pytest.raises(ValueError, match="not in the table"):
        season.fixture_slots(tab, ["A"], ["D"], known_teams=["A", "B", "C", "D"])
    with pytest.raises(ValueError, match="plays itself"):
        season.fixture_slots(tab, ["A"], ["A"])
    with pytest.raises(ValueError, match="at most 64"):
        season.build_table([f"T{i}" for i in range(65)])
    for bad in ((3, 4), (0, 0), (3.0, 1), (3, -1), (True, 0), "ab", (3,)):
        with pytest.raises(ValueError, match="points"):
            season.build_table(["A", "B"], points=bad)
    with pytest.raises(ValueError, match="not in the table"):
        season.build_table(["A", "B"], {"home_team": ["A"], "away_team": ["C"], "home_goals": [1], "away_goals": [0]})
    assert season.table_teams(["B", "A"], ["C", "A"], {"home_team": ["D"], "away_team": ["A"]}) == ["A", "B", "C", "D"]


def test_groups_and_probabilities():
    """Group labels map to sorted ids; P is the largest group; counts turn into probabilities and expected points."""
    tab = season.build_table(["A", "B", "C", "D", "E"], groups={"A": "y", "B": "x", "C": "y", "D": "x", "E": "y"})
    assert tab["group_labels"] == ["x", "y"]
    np.testing.assert_array_equal(tab["group"], [1, 0, 1, 0, 1])
    season.fixture_slots(tab, ["A", "B"], ["C", "D"])
    assert tab["num_positions"] == 3 and tab["num_points_bins"] == 4
    pc = np.array([[2, 2, 0]] * 5)
    bc = np.array([[1, 1, 0, 2]] * 5)
    pr = season.probabilities(tab, pc, bc, 4)
    np.testing.assert_allclose(pr["position_proba"].sum(axis=1), 1.0)
    np.testing.assert_allclose(pr["expected_points"], (0 * 1 + 1 * 1 + 3 * 2) / 4)
