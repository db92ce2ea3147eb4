"""Pairings drawn by lot on the CPU: season.build_bracket with pairings and its refusals, the ctypes struct and prototypes
against include/bplx.h, the oracle's open and seeded procedures on hand-worked pools, the exact distribution of the
seeded procedure against a brute-force walk of its tree, and a protected 8 + 8 pool where the sequential procedure is
not a uniform choice among the valid pairings."""
import ctypes as C
import itertools
import re
from fractions import Fraction

import numpy as np
import pytest

from bpl_next_b200 import _abi, season
from oracle import pairing as op


def _uefa_table():
    teams = [f"T{i:02d}" for i in range(32)]
    groups = {t: "ABCDEFGH"[i // 4] for i, t in enumerate(teams)}
    return teams, groups, season.build_table(teams, groups=groups)


def _uefa_ties(protect=("group", "association")):
    """A seeded round of 16 (winners against runners-up), open quarter- and semi-final draws, a final."""
    L = "ABCDEFGH"
    pairings = [{"id": "r16", "pool": [("group", g, 0) for g in L] + [("group", g, 1) for g in L],
                 "pots": [0] * 8 + [1] * 8, "protect": set(protect), "seeded_home": False},
                {"id": "qf", "pool": [("winner", f"r16_{i}") for i in range(8)], "pots": None},
                {"id": "sf", "pool": [("winner", f"qf_{i}") for i in range(4)], "pots": None}]
    ties = [{"id": f"r16_{i}", "round": "R16", "pair": ("r16", i), "format": "two_legs"} for i in range(8)]
    ties += [{"id": f"qf_{i}", "round": "QF", "pair": ("qf", i), "format": "two_legs"} for i in range(4)]
    ties += [{"id": f"sf_{i}", "round": "SF", "pair": ("sf", i), "format": "two_legs"} for i in range(2)]
    ties += [{"id": "final", "round": "F", "home": ("winner", "sf_0"), "away": ("winner", "sf_1"),
              "format": "extra_time", "neutral_venue": 1}]
    return pairings, ties


def test_build_bracket_with_pairings():
    teams, groups, tab = _uefa_table()
    pairings, ties = _uefa_ties()
    assoc = {t: f"N{i % 5}" for i, t in enumerate(teams)}
    assoc["T31"] = None
    br = season.build_bracket(tab, ties, pairings=pairings, association=assoc)
    assert br["pairing_ids"] == ["r16", "qf", "sf"]
    np.testing.assert_array_equal(br["pairing_mode"], [_abi.PAIRING_SEEDED, _abi.PAIRING_OPEN, _abi.PAIRING_OPEN])
    np.testing.assert_array_equal(br["pairing_protect"], [3, 0, 0])
    np.testing.assert_array_equal(br["pairing_host_pot"], [1, 0, 0])
    np.testing.assert_array_equal(br["pool_size"], [16, 8, 4])
    assert br["pool_kind"].shape == (3, 64)
    np.testing.assert_array_equal(br["pool_kind"][0, :16], _abi.ENTRANT_GROUP_POS)
    np.testing.assert_array_equal(br["pool_arg0"][0, :16], list(range(8)) * 2)
    np.testing.assert_array_equal(br["pool_arg1"][0, :16], [0] * 8 + [1] * 8)
    np.testing.assert_array_equal(br["pool_pot"][0, :16], [0] * 8 + [1] * 8)
    np.testing.assert_array_equal(br["pool_kind"][1, :8], _abi.ENTRANT_WINNER)
    np.testing.assert_array_equal(br["pool_arg0"][1, :8], np.arange(8))
    np.testing.assert_array_equal(br["kind"][:14], _abi.ENTRANT_PAIRED)
    np.testing.assert_array_equal(br["arg0"][8:12], 1)
    np.testing.assert_array_equal(br["arg1"][8:12], [[0, 1], [2, 3], [4, 5], [6, 7]])
    np.testing.assert_array_equal(br["kind"][14], _abi.ENTRANT_WINNER)
    assert br["slot_assoc"][31] == 0xFF and br["slot_assoc"][0] == 0 and br["slot_assoc"][6] == 1
    np.testing.assert_array_equal(br["tie_format"], [2] * 14 + [1])
    # no pairings: the bracket of before, without pairing keys
    plain = season.build_bracket(tab, [{"id": "f", "round": "F", "home": ("group", "A", 0), "away": ("group", "B", 0)}])
    assert "pool_kind" not in plain


def _refuse(match, **change):
    teams, groups, tab = _uefa_table()
    pairings, ties = _uefa_ties(protect=())
    assoc = None
    if "pairings" in change:
        pairings = change["pairings"](pairings)
    if "ties" in change:
        ties = change["ties"](ties)
    if "table" in change:
        tab = change["table"](tab)
    if "association" in change:
        assoc = change["association"]
    with pytest.raises(ValueError, match=match):
        season.build_bracket(tab, ties, pairings=pairings, association=assoc)


def _set(i, **kv):
    def f(pg):
        pg = [dict(p) for p in pg]
        pg[i].update(kv)
        return pg
    return f


def test_build_bracket_pairing_refusals():
    _refuse("even pool", pairings=_set(2, pool=[("winner", f"qf_{i}") for i in range(3)]),
            ties=lambda t: t[:12] + [dict(t[12], pair=("sf", 0))] + [t[14]])
    _refuse("equal in size", pairings=_set(0, pots=[0] * 9 + [1] * 7))
    _refuse("0 or 1", pairings=_set(0, pots=[0] * 8 + [2] * 8))
    _refuse("protections need a seeded draw", pairings=_set(1, protect={"group"}))
    _refuse("unknown protection", pairings=_set(0, protect={"fair_play"}))
    _refuse("association protection needs association", pairings=_set(0, protect={"association"}))
    _refuse("group protection needs a table with groups", pairings=_set(0, protect={"group"}),
            table=lambda tab: season.build_table(tab["teams"]),
            ties=lambda t: t)
    _refuse("at most 16 pairings", pairings=lambda pg: pg + [dict(pg[2], id=f"x{i}") for i in range(14)])
    teams, groups, tab = _uefa_table()
    with pytest.raises(ValueError, match="1 of its pairs feed no tie"):
        season.build_bracket(tab, [{"id": "a", "round": "R1", "pair": ("p", 0)},
                                   {"id": "f", "round": "F", "home": ("winner", "a"), "away": ("group", "B", 0)}],
                             pairings=[{"id": "p", "pool": [("group", g, 0) for g in "ADCE"], "pots": None}])
    _refuse("taken twice", ties=lambda t: t[:7] + [dict(t[7], pair=("r16", 6))] + t[8:])
    _refuse("has no pair 8", ties=lambda t: t[:7] + [dict(t[7], pair=("r16", 8))] + t[8:])
    _refuse("unknown pairing", ties=lambda t: t[:7] + [dict(t[7], pair=("r32", 7))] + t[8:])
    _refuse("not played before", pairings=_set(1, pool=[("winner", f"r16_{i}") for i in range(7)] + [("winner", "qf_3")]))
    _refuse("used twice", pairings=_set(1, pool=[("winner", "r16_0")] * 8))
    _refuse("unknown entrant", pairings=_set(1, pool=[("paired", "r16", 0)] + [("winner", f"r16_{i}") for i in range(1, 8)]))
    _refuse("pair or a home", ties=lambda t: [dict(t[0], home=("group", "A", 0))] + t[1:])
    _refuse("labels", pairings=_set(0, protect={"association"}), association=["x"] * 3)


def test_struct_and_prototypes_match_the_header():
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} bplx_pairings;", text).group(1)
    fields = re.findall(r"(\w+);", re.sub(r"/\*.*?\*/", "", body))
    assert [f[0] for f in _abi.Pairings._fields_] == fields
    assert C.sizeof(_abi.Pairings) == 8 + 9 * 8 and _abi.Pairings.mode.offset == 8
    for name, value in (("BPLX_ENTRANT_PAIRED", _abi.ENTRANT_PAIRED), ("BPLX_MAX_PAIRINGS", _abi.MAX_PAIRINGS),
                        ("BPLX_PAIRING_MAX_POOL", _abi.PAIRING_MAX_POOL), ("BPLX_PAIRING_MAX_POT", _abi.PAIRING_MAX_POT),
                        ("BPLX_PAIRING_OPEN", _abi.PAIRING_OPEN), ("BPLX_PAIRING_SEEDED", _abi.PAIRING_SEEDED),
                        ("BPLX_PROTECT_GROUP", _abi.PROTECT_GROUP),
                        ("BPLX_PROTECT_ASSOCIATION", _abi.PROTECT_ASSOCIATION)):
        assert re.search(rf"#define {name} (\d+)", text).group(1) == str(value), name
    class Stub:  # takes argtypes / restypes of any symbol: no library needed
        def __getattr__(self, name):
            f = type("F", (), {})()
            setattr(self, name, f)
            return f

    lib = _abi.declare(Stub())
    for fn in ("bplx_simulate_tournament_paired", "bplx_simulate_tournament_paired_workspace_bytes"):
        decl = re.search(rf"\b{fn}\(([^;]*)\);", text).group(1)
        assert len(getattr(lib, fn).argtypes) == decl.count(",") + 1, fn
    args = getattr(lib, "bplx_simulate_tournament_paired").argtypes
    assert args[7] == C.POINTER(_abi.Ranking) and args[8] == C.POINTER(_abi.Pairings)


def test_open_draw_by_hand():
    top = 0xFFFFFFFF
    assert op.open_draw("ABCD", [0, 0, 0]) == [("A", "B"), ("C", "D")]
    # i = 0: j = 3 -> DBCA; i = 1: j = 3 -> DACB; i = 2: j = 3 -> DABC
    assert op.open_draw("ABCD", [top, top, top]) == [("D", "A"), ("B", "C")]
    # i = 0: j = 0 + (2^31 * 4 >> 32) = 2 -> CBAD
    assert op.open_draw("ABCD", [1 << 31, 0, 0]) == [("C", "B"), ("A", "D")]
    assert op.index(top, 5) == 4 and op.index(0, 5) == 0 and op.index(1 << 31, 5) == 2


def test_seeded_draw_by_hand():
    # a0 may not meet b0: b0 drawn first must take a1
    assert op.seeded_draw([[False, True], [True, True]], [0, 0, 0, 0]) == [(1, 0), (0, 1)]
    # b0 may meet a0 and a1, b1 only a0, b2 only a2: with b0 drawn first a0 would strand b1, so only a1 is eligible,
    # whatever w_1 says
    compat = [[True, True, False], [True, False, False], [False, False, True]]
    for w1 in (0, 0xFFFFFFFF):
        assert op.seeded_draw(compat, [0, w1, 0, 0, 0, 0]) == [(1, 0), (0, 1), (2, 2)]
    # nothing may meet b2 at all: no pairing
    assert op.seeded_draw([[True, True, False]] * 3, [0] * 6) is None
    assert op.seeded_pair_proba([[True, True, False]] * 3) is None


def _tree(compat, ra, rb, p, out):
    """The procedure's tree walked explicitly, with exact fractions (no memo, no masks)."""
    if not rb:
        return
    for b in rb:
        rb2 = [x for x in rb if x != b]
        elig = [a for a in ra if compat[a][b] and op._feasible([x for x in ra if x != a], rb2, compat)]
        for a in elig:
            q = p / len(rb) / len(elig)
            out[a][b] += q
            _tree(compat, [x for x in ra if x != a], rb2, q, out)


def test_dynamic_program_against_the_procedure_tree():
    rng = np.random.default_rng(3)
    for _ in range(6):
        compat = (rng.random((4, 4)) < 0.6).tolist()
        dp = op.seeded_pair_proba(compat, Fraction(1))
        if dp is None:
            assert not op._feasible(range(4), range(4), compat)
            continue
        tree = [[Fraction(0)] * 4 for _ in range(4)]
        _tree(compat, list(range(4)), list(range(4)), Fraction(1), tree)
        assert dp == tree
        assert all(sum(row) == 1 for row in dp) and all(sum(col) == 1 for col in zip(*dp))
        assert all(dp[a][b] == 0 for a in range(4) for b in range(4) if not compat[a][b])


def protected_8_8():
    """Group winners (pot A) against runners-up (pot B) of 8 groups, group protection (a_g never meets b_g) and
    association protection with three associations among them: slot g is group g's winner, 8 + g its runner-up."""
    group = list(range(8)) * 2
    assoc = [0, 2, 2, 2, 0, 2, 1, 0] + [1, 2, 0, 1, 0, 0, 2, 0]
    return group, assoc, op.compat_matrix(list(range(8)), list(range(8, 16)), 3, group, assoc)


# the GPU test's tolerance for pair probabilities: 5 sigma at N = 2^22 and p = 1/2 (the largest sigma)
GPU_TOLERANCE = 5 * np.sqrt(0.25 / 2 ** 22)


def test_sequential_procedure_is_not_uniform_over_valid_pairings():
    _, _, compat = protected_8_8()
    seq, uni = np.array(op.seeded_pair_proba(compat)), np.array(op.uniform_pair_proba(compat))
    np.testing.assert_allclose(seq.sum(axis=0), 1, atol=1e-12)
    np.testing.assert_allclose(seq.sum(axis=1), 1, atol=1e-12)
    assert (seq[~np.array(compat)] == 0).all()
    assert np.abs(seq - uni).max() > 10 * GPU_TOLERANCE, np.abs(seq - uni).max()


def test_open_draw_pairs_every_two_entrants_with_one_over_n_minus_one():
    """Every sequence of Fisher-Yates choices (j_i uniform over n - i) of a pool of 6: each unordered pair meets in
    exactly 1/5 of them, and each entrant is at home in exactly half."""
    n = 6
    meet, home = np.zeros((n, n), np.int64), np.zeros(n, np.int64)
    seqs = list(itertools.product(*[range(n - i) for i in range(n - 1)]))
    for js in seqs:
        words = [((j << 32) + (n - i) - 1) // (n - i) for i, j in enumerate(js)]  # the smallest w with index j
        assert [op.index(w, n - i) for i, w in enumerate(words)] == list(js)
        for h, a in op.open_draw(range(n), words):
            meet[h, a] += 1
            home[h] += 1
    both = meet + meet.T
    off = ~np.eye(n, dtype=bool)
    assert (both[off] * (n - 1) == len(seqs)).all() and (home * 2 * n == len(seqs) * n).all()
