"""Knockout tie formats on the CPU: ``season.build_bracket``'s ``format`` key and refusals, the ctypes prototype and
constants against the header, ``resolve_bracket`` on hand-made two-legged, extra-time and penalty ties, and the float64
oracle's sampler against its own closed form (P(A through), P(extra time), P(penalties) per draw)."""
import ctypes as C
import re

import numpy as np
import pytest

from bpl_next_b200 import _abi, season
from oracle import tournament
from tests.test_score_grid_gpu import make_samples
from tests.test_tournament import _euro


def test_build_bracket_formats():
    tab, ties = _euro()
    best = {"position": 2, "count": 4}
    plain = season.build_bracket(tab, ties, best)
    np.testing.assert_array_equal(plain["tie_format"], np.zeros(len(ties), np.uint8))
    fmt = [dict(t) for t in ties]
    for t in fmt[:8]:
        t["format"] = "two_legs"
    for t in fmt[8:12]:
        t["format"] = "one_match"
    fmt[-1]["format"] = "extra_time"  # the final, at a neutral venue
    b = season.build_bracket(tab, fmt, best)
    assert b["tie_format"].dtype == np.uint8
    np.testing.assert_array_equal(b["tie_format"], [_abi.TIE_TWO_LEGS] * 8 + [_abi.TIE_ONE_MATCH] * 6
                                  + [_abi.TIE_ONE_MATCH_ET])
    # every key a bracket without formats had is unchanged
    assert set(b) == set(plain)
    for k, v in plain.items():
        if k != "tie_format":
            np.testing.assert_array_equal(np.asarray(b[k], dtype=object), np.asarray(v, dtype=object), err_msg=k)
    pr = season.bracket_probabilities(b, np.zeros((24, 4)), np.zeros((24, 4)), 1, np.ones((15, 3)))
    assert pr["tie_ids"] == b["ids"] and pr["decided_proba"].shape == (15, 3)


def test_build_bracket_format_refusals():
    tab, ties = _euro()
    bad = [dict(t) for t in ties]
    bad[0]["format"] = "golden_goal"
    with pytest.raises(ValueError, match="unknown format"):
        season.build_bracket(tab, bad, {"position": 2, "count": 4})
    bad = [dict(t) for t in ties]
    bad[-1]["format"] = "two_legs"  # the final is at a neutral venue
    with pytest.raises(ValueError, match="two-legged tie cannot be at a neutral venue"):
        season.build_bracket(tab, bad, {"position": 2, "count": 4})


def test_prototype_and_constants_match_the_header():
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    for name, val in (("BPLX_TIE_ONE_MATCH", _abi.TIE_ONE_MATCH), ("BPLX_TIE_ONE_MATCH_ET", _abi.TIE_ONE_MATCH_ET),
                      ("BPLX_TIE_TWO_LEGS", _abi.TIE_TWO_LEGS)):
        assert f"#define {name} {val}" in text
    assert "#define BPLX_EXTRA_TIME_FRACTION (1.0 / 3.0)" in text and _abi.EXTRA_TIME_FRACTION == 1.0 / 3.0
    assert season.TIE_FORMATS == {"one_match": 0, "extra_time": 1, "two_legs": 2}
    proto = re.search(r"int bplx_simulate_tournament_ex\(([^;]*)\);", text).group(1)
    params = [p.strip() for p in proto.split(",")]
    fn = _abi.lib().bplx_simulate_tournament_ex
    assert len(fn.argtypes) == len(params) == 26 and fn.restype == C.c_int
    # bplx_simulate_tournament's arguments, plus tie_format after the bracket, decided_counts after win_counts and
    # ko_extra after ko_winners
    old = re.search(r"int bplx_simulate_tournament\(([^;]*)\);", text).group(1)
    names = [re.split(r"[ *]+", p.strip())[-1] for p in params]
    old_names = [re.split(r"[ *]+", p.strip())[-1] for p in old.split(",")]
    assert [n for n in names if n not in ("tie_format", "decided_counts", "ko_extra")] == old_names
    assert names.index("tie_format") == names.index("b") + 1
    assert names.index("decided_counts") == names.index("win_counts") + 1
    assert names.index("ko_extra") == names.index("ko_winners") + 1


def _cup():
    """Four teams, no group stage: two two-legged semi-finals, a third-place match with extra time, a one-match
    final."""
    names = ["A", "B", "C", "D"]
    tab = season.build_table(names)
    season._size_histograms(tab)
    ties = [{"id": "s1", "round": "SF", "home": ("team", "A"), "away": ("team", "B"), "format": "two_legs"},
            {"id": "s2", "round": "SF", "home": ("team", "C"), "away": ("team", "D"), "format": "two_legs"},
            {"id": "3rd", "round": "third", "home": ("loser", "s1"), "away": ("loser", "s2"), "format": "extra_time"},
            {"id": "f", "round": "F", "home": ("winner", "s1"), "away": ("winner", "s2")}]
    return tab, season.build_bracket(tab, ties)


def test_resolve_bracket_by_hand():
    """s1: A-B 1-1, then B-A 2-2 (level on aggregate), extra time in leg 2 0-0, B wins the shoot-out; s2: C-D 0-2,
    then D-C 0-3 (C through on aggregate, won in leg 2); third place A-D 1-1, A scores in extra time; final B-C 0-0,
    the lot to B.  The loser of the shoot-out, A, reaches the third-place match."""
    tab, b = _cup()
    X = tournament.NOT_PLAYED
    e = np.zeros((1, 0), np.int64)
    keys = np.zeros((1, 4), np.int64)
    ko_h, ko_a = np.array([[1, 0, 1, 0]]), np.array([[1, 2, 1, 0]])
    extra = np.array([[[2, 2, 0, 0], [3, 0, X, X], [X, X, 1, 0], [X, X, X, X]]])
    through = np.array([[0, 1, 1, 1]])  # read only where the tie is level after everything else
    r = tournament.resolve_bracket(tab, e[0], e[0], b, e, e, keys, ko_h, ko_a, through, ko_extra=extra)
    A, B, C_, D = range(4)
    np.testing.assert_array_equal(r["ko_entrants"][0], [[A, B], [C_, D], [A, D], [B, C_]])
    np.testing.assert_array_equal(r["ko_winners"][0], [B, C_, A, B])
    np.testing.assert_array_equal(r["ko_extra"], extra)
    np.testing.assert_array_equal(r["decided_counts"], [[0, 0, 1], [1, 0, 0], [0, 1, 0], [0, 0, 1]])
    np.testing.assert_array_equal(r["reach_counts"], [[1, 1, 0], [1, 0, 1], [1, 0, 1], [1, 1, 0]])
    np.testing.assert_array_equal(r["win_counts"], [[0, 1, 0], [1, 0, 1], [1, 0, 0], [0, 0, 0]])
    # the same scores, B losing the shoot-out instead: A goes through and meets C in the final
    through2 = np.array([[1, 1, 1, 1]])
    r2 = tournament.resolve_bracket(tab, e[0], e[0], b, e, e, keys, ko_h, ko_a, through2, ko_extra=extra)
    np.testing.assert_array_equal(r2["ko_entrants"][0], [[A, B], [C_, D], [B, D], [A, C_]])
    # settle: a two-legged tie won on aggregate although its first leg was lost
    th, how = tournament.settle(tournament.TWO_LEGS, np.array([0]), np.array([2]), np.array([[3, 0, X, X]]),
                                np.array([False]))
    assert th[0] and how[0] == 0


@pytest.mark.parametrize("model,fmt,neutral", [("dixon_coles", tournament.TWO_LEGS, 0),
                                               ("neutral_wc", tournament.ONE_MATCH_ET, 1),
                                               ("neutral", tournament.TWO_LEGS, 0)])
def test_oracle_sampler_against_its_closed_form(model, fmt, neutral):
    """One tie at N = 2e5 (50 draws x 4,000): the oracle's shares of A through, extra time and penalties are within
    5 sigma of the mean over draws of ``tie_closed_form``; its decided counts add up to N."""
    S, R, G = 50, 4000, 15
    N = S * R
    s = {k: v.astype(np.float64) for k, v in make_samples(model, S, 4, 3, seed=31).items()}
    tab = season.build_table(["P", "Q"])
    season._size_histograms(tab)
    tie = {"id": "t", "round": "F", "home": ("team", "P"), "away": ("team", "Q"), "neutral_venue": neutral,
           "format": {tournament.ONE_MATCH_ET: "extra_time", tournament.TWO_LEGS: "two_legs"}[fmt]}
    br = season.build_bracket(tab, [tie])
    br["slot_team"] = np.array([2, 0], np.uint16)
    br["slot_conf"] = np.array([1, 2], np.uint8)
    e = np.zeros(0, np.uint8)
    o = tournament.simulate_tournament(model, s, None, e, e, tab, br, G, R, seed=5)
    assert o["invalid"] == 0
    dec = o["decided_counts"][0]
    assert dec.sum() == N
    p_through, p_et, p_pen = (x.mean() for x in tournament.tie_closed_form(model, s, 2, 0, fmt, G, neutral, 1, 2))
    for share, p in (((o["ko_winners"][:, 0] == 0).mean(), p_through), (dec[1:].sum() / N, p_et),
                     (dec[2] / N, p_pen)):
        assert abs(share - p) <= 5 * np.sqrt(p * (1 - p) / N), (share, p)
    played = o["ko_extra"][:, 0, 2] != tournament.NOT_PLAYED
    assert played.sum() == dec[1:].sum()
    if fmt == tournament.ONE_MATCH_ET:
        assert (o["ko_extra"][:, 0, :2] == tournament.NOT_PLAYED).all()
