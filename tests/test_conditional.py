"""Match importance on the CPU: season.build_conditions and its refusals, the ctypes struct and prototype against
include/bplx.h, oracle/conditional.py against a brute-force loop and the two identities, and
season.conditional_probabilities on hand-made counts."""
import ctypes as C
import re

import numpy as np
import pytest

from bpl_next_b200 import _abi, season
from oracle import conditional as oc
from oracle import simulate as osim
from tests.test_score_grid_gpu import make_samples


def _groups_table():
    teams = [f"T{i}" for i in range(8)]
    groups = {t: "AB"[i % 2] for i, t in enumerate(teams)}  # A: T0 T2 T4 T6, B: T1 T3 T5 T7
    return season.build_table(teams, groups=groups)


def test_build_conditions_maps_teams_positions_and_labels():
    tab = _groups_table()
    c = season.build_conditions(tab, 12, [7, 3, 11], {"T5 wins B": ("T5", 0), "T2 through": ("T2", range(2)),
                                                      "T7 last": ("T7", [3])})
    assert c["key_fixtures"] == [7, 3, 11] and c["events"] == ["T5 wins B", "T2 through", "T7 last"]
    np.testing.assert_array_equal(c["event_slot"], [5, 2, 7])
    np.testing.assert_array_equal(c["event_positions"], np.asarray([1, 3, 8], np.uint64))
    assert c["event_positions"].dtype == np.uint64 and c["event_slot"].dtype == np.uint8
    (g,) = c["groups"]
    np.testing.assert_array_equal(g["key_fixture"], [3, 7, 11])
    np.testing.assert_array_equal(g["rows"], [1, 0, 2])
    assert g["key_fixture"].dtype == np.int32


def test_build_conditions_groups_more_than_64_keys():
    tab = season.build_table([f"T{i}" for i in range(20)])
    rng = np.random.default_rng(1)
    keys = rng.permutation(380)[:150].tolist()
    c = season.build_conditions(tab, 380, keys, {"title": ("T3", 0)})
    assert [len(g["key_fixture"]) for g in c["groups"]] == [64, 64, 22]
    flat = np.concatenate([g["key_fixture"] for g in c["groups"]])
    np.testing.assert_array_equal(flat, np.sort(keys))
    for g in c["groups"]:
        assert (np.diff(g["key_fixture"]) > 0).all()
        np.testing.assert_array_equal(np.asarray(keys)[g["rows"]], g["key_fixture"])
    # rows cover the caller's order exactly once
    np.testing.assert_array_equal(np.sort(np.concatenate([g["rows"] for g in c["groups"]])), np.arange(150))
    # relegation of a 20-team league
    c = season.build_conditions(tab, 380, [0], {"down": ("T0", (17, 18, 19))})
    assert int(c["event_positions"][0]) == (1 << 17) | (1 << 18) | (1 << 19)


@pytest.mark.parametrize("keys,events,match", [
    ([], {"e": ("T0", 0)}, "empty"),
    ([12], {"e": ("T0", 0)}, "not one of the 12"),
    ([-1], {"e": ("T0", 0)}, "not one of the 12"),
    ([3, 3], {"e": ("T0", 0)}, "more than once"),
    ([3], {}, "between 1 and 64"),
    ([3], {f"e{i}": ("T0", 0) for i in range(65)}, "between 1 and 64"),
    ([3], {"e": ("X", 0)}, "not in the table"),
    ([3], {"e": ("T0", 4)}, "group of 4"),
    ([3], {"e": ("T0", -1)}, "group of 4"),
    ([3], {"e": ("T0", [])}, "no positions"),
    ([3], {"e": ("T0", [True])}, "group of 4"),
    ([3], {"e": ("T0", 0, 1)}, "expected \\(team, positions\\)"),
])
def test_build_conditions_refusals(keys, events, match):
    with pytest.raises(ValueError, match=match):
        season.build_conditions(_groups_table(), 12, keys, events)


def test_struct_and_prototype_match_the_header():
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} bplx_conditions;", text).group(1)
    fields = re.findall(r"(\w+);", re.sub(r"/\*.*?\*/", "", body))
    assert [f[0] for f in _abi.Conditions._fields_] == fields
    assert C.sizeof(_abi.Conditions) == 40 and _abi.Conditions.event_positions.offset == 32
    for name, value in (("BPLX_SIM_MAX_KEY_FIXTURES", _abi.SIM_MAX_KEY_FIXTURES),
                        ("BPLX_SIM_MAX_EVENTS", _abi.SIM_MAX_EVENTS)):
        assert re.search(rf"#define {name} (\d+)", text).group(1) == str(value), name

    class Stub:  # takes argtypes / restypes of any symbol: no library needed
        def __getattr__(self, name):
            f = type("F", (), {})()
            setattr(self, name, f)
            return f

    lib = _abi.declare(Stub())
    decl = re.search(r"\bbplx_simulate_table_conditional\(([^;]*)\);", text).group(1)
    args = lib.bplx_simulate_table_conditional.argtypes
    assert len(args) == decl.count(",") + 1 == len(lib.bplx_simulate_table_ex.argtypes) + 3
    assert args[5] == C.POINTER(_abi.Ranking) and args[6] == C.POINTER(_abi.Conditions)


def _brute(home, away, positions, valid, keys, slots, masks):
    Kc, E = len(keys), len(slots)
    o, c = np.zeros((Kc, 3), np.int64), np.zeros((Kc, 3, E), np.int64)
    for i in range(len(valid)):
        if not valid[i]:
            continue
        for j, f in enumerate(keys):
            h, a = int(home[i, f]), int(away[i, f])
            out = 0 if h > a else 1 if h == a else 2
            o[j, out] += 1
            for e, (t, m) in enumerate(zip(slots, masks)):
                if (int(m) >> int(positions[i, t])) & 1:
                    c[j, out, e] += 1
    return o, c


def _oracle_case(model="dixon_coles", S=40, R=3, T=8, F=30, seed=5, grouped=True):
    s = make_samples(model, S, T + 2, 4, seed=seed)
    rng = np.random.default_rng(seed)
    names = [f"T{i}" for i in range(T)]
    tab = season.build_table(names, groups=[f"g{i % 2}" for i in range(T)] if grouped else None)
    h = rng.integers(0, T, F)
    a = (h + rng.integers(1, T, F)) % T
    hs, as_ = season.fixture_slots(tab, [names[i] for i in h], [names[i] for i in a])
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16)}
    return s, fx, hs, as_, tab


def test_oracle_counts_against_a_brute_force_loop_and_the_identities():
    s, fx, hs, as_, tab = _oracle_case()
    o = osim.simulate("dixon_coles", s, fx, hs, as_, tab, 10, 3, 17)
    rng = np.random.default_rng(2)
    valid = o["valid"].copy()
    valid[::7] = False  # (some simulations left out, as invalid ones are)
    keys = np.sort(rng.permutation(30)[:9])
    slots = rng.integers(0, 8, 11).astype(np.uint8)
    masks = rng.integers(1, 16, 11).astype(np.uint64)
    got = oc.counts(o["home"], o["away"], o["positions"], valid, keys, slots, masks)
    want = _brute(o["home"], o["away"], o["positions"], valid, keys, slots, masks)
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)
    # the identities, with the histograms of the same simulations
    hist = osim.histograms(tab, osim.tables(tab, hs, as_, o["home"], o["away"])[0], o["positions"], valid)
    pc = hist["position_counts"]
    for j in range(len(keys)):
        assert got[0][j].sum() == valid.sum()
        for e, (t, m) in enumerate(zip(slots, masks)):
            assert got[1][j, :, e].sum() == sum(pc[t, p] for p in range(pc.shape[1]) if (int(m) >> p) & 1)
    # oracle.conditional.simulate: the same counts from the replay, under either rule
    cond = {"key_fixture": keys, "event_slot": slots, "event_positions": masks}
    full = oc.simulate("dixon_coles", s, fx, hs, as_, tab, 10, 3, 17, cond)
    want = _brute(full["home"], full["away"], full["positions"], full["valid"], keys, slots, masks)
    np.testing.assert_array_equal(full["outcome_counts"], want[0])
    np.testing.assert_array_equal(full["conditional_counts"], want[1])
    hh = oc.simulate("dixon_coles", s, fx, hs, as_, tab, 10, 3, 17, cond, tiebreak="head_to_head")
    want = _brute(hh["home"], hh["away"], hh["positions"], hh["valid"], keys, slots, masks)
    np.testing.assert_array_equal(hh["conditional_counts"], want[1])


def test_conditional_probabilities_on_hand_made_counts():
    cond = {"key_fixtures": [4, 1, 9], "events": ["title", "down"]}
    # fixture 4: all three outcomes; fixture 1: only home wins and draws; fixture 9: only home wins
    o = np.array([[50, 30, 20], [60, 40, 0], [100, 0, 0]])
    c = np.zeros((3, 3, 2), np.int64)
    c[0, :, 0] = (25, 6, 1)
    c[0, :, 1] = (5, 6, 10)
    c[1, :, 0] = (20, 12, 0)
    c[1, :, 1] = (6, 15, 0)
    c[2, :, 0] = (32, 0, 0)
    c[2, :, 1] = (21, 0, 0)
    r = season.conditional_probabilities(cond, o, c, 100)
    assert r["key_fixtures"] == [4, 1, 9] and r["events"] == ["title", "down"]
    np.testing.assert_allclose(r["outcome_proba"], o / 100)
    np.testing.assert_allclose(r["event_proba"], [0.32, 0.21])
    np.testing.assert_allclose(r["conditional_proba"][0, :, 0], [0.5, 0.2, 0.05])
    np.testing.assert_allclose(r["conditional_proba"][1, :2, 1], [0.1, 0.375])
    assert np.isnan(r["conditional_proba"][1, 2]).all() and np.isnan(r["conditional_proba"][2, 1:]).all()
    np.testing.assert_allclose(r["importance"][0], [0.45, 0.4])
    np.testing.assert_allclose(r["importance"][1], [1 / 3 - 0.3, 0.275])
    np.testing.assert_array_equal(r["importance"][2], [0.0, 0.0])
    np.testing.assert_array_equal(r["outcome_counts"], o)
    np.testing.assert_array_equal(r["conditional_counts"], c)
