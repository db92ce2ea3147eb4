"""CPU: the float64 market reference against a grid written out by hand, its means against the averaged predict grid,
the refusals of predict_proba_posterior (before any GPU work) and the ctypes mirror of bplx_market_lines."""
import ctypes as C
import math
import re

import numpy as np
import pytest

from bpl_next_b200 import _abi
from oracle import markets as om
from oracle import predict as op
from tests.test_score_grid_gpu import make_fixtures, make_samples


def _pois(k, lam):
    return math.exp(-lam) * lam ** k / math.factorial(k)


def test_oracle_rows_by_hand_on_a_two_goal_grid():
    # Dixon-Coles, teams 0 (home) and 1, two draws; draw 1's c makes tau(0, 0) = 1 - c lh la negative: clamped to 0
    s = {"attack": np.array([[0.2, -0.1], [0.5, 0.0]]), "defence": np.array([[0.1, 0.3], [-0.2, 0.1]]),
         "home_advantage": np.array([0.25, 0.1]), "corr_coef": np.array([-0.1, 0.9])}
    tl, ml = (1.5, 2.5, 3.5), (-1.5, 1.5)
    got = om.market_draws("dixon_coles", s, [0], [1], 2, tl, ml)[:, 0, :]
    names = om.market_names(tl, ml)
    cells = {(i, j) for i in range(3) for j in range(3)}
    rows = {"home_win": {(1, 0), (2, 0), (2, 1)}, "draw": {(0, 0), (1, 1), (2, 2)}, "away_win": {(0, 1), (0, 2), (1, 2)},
            "both_teams_score": {(1, 1), (1, 2), (2, 1), (2, 2)},
            "total_over_1.5": {(0, 2), (1, 1), (2, 0), (1, 2), (2, 1), (2, 2)},
            "total_under_1.5": {(0, 0), (0, 1), (1, 0)},
            "total_over_2.5": {(1, 2), (2, 1), (2, 2)},
            "total_under_2.5": {(0, 0), (0, 1), (1, 0), (0, 2), (1, 1), (2, 0)},
            "total_over_3.5": {(2, 2)}, "total_under_3.5": cells - {(2, 2)},
            "home_margin_over_-1.5": cells - {(0, 2)}, "home_margin_under_-1.5": {(0, 2)},
            "home_margin_over_1.5": {(2, 0)}, "home_margin_under_1.5": cells - {(2, 0)}}
    for d in range(2):
        lh = math.exp(s["attack"][d, 0] - s["defence"][d, 1] + s["home_advantage"][d])
        la = math.exp(s["attack"][d, 1] - s["defence"][d, 0])
        c = s["corr_coef"][d]
        tau = {(0, 0): max(1 - c * lh * la, 0.0), (0, 1): max(1 + c * lh, 0.0), (1, 0): max(1 + c * la, 0.0),
               (1, 1): max(1 - c, 0.0)}
        if d == 1:
            assert 1 - c * lh * la < 0 and tau[(0, 0)] == 0.0
        P = {(i, j): tau.get((i, j), 1.0) * _pois(i, lh) * _pois(j, la) for (i, j) in cells}
        want = {name: sum(P[x] for x in cl) for name, cl in rows.items()}
        want.update(home_rate=lh, away_rate=la)
        assert sorted(want) == sorted(names)
        for k, name in enumerate(names):
            assert abs(got[d, k] - want[name]) <= 1e-15, (d, name, got[d, k], want[name])
    # the mass beyond max_goals is dropped: over and under of a line do not sum to 1
    assert (got[:, names.index("total_over_2.5")] + got[:, names.index("total_under_2.5")] < 1).all()


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
def test_oracle_means_are_the_averaged_grid(model):
    S, T, F, Cf, mg = 40, 6, 9, 3, 8
    s = make_samples(model, S, T, Cf, seed=11)
    fx = make_fixtures(model, F, T, Cf, seed=12)
    kw = {k: fx[k] for k in ("home_conf", "away_conf", "neutral_venue") if k in fx}
    tl, ml = (0.5, 2.5, 15.5), (-7.5, -0.5, 0.5, 3.5)
    v = om.market_draws(model, s, fx["home_team"], fx["away_team"], mg, tl, ml, **kw).mean(axis=0)
    grid, _, _ = op.predict_score_grid_proba(model, s, fx["home_team"], fx["away_team"], mg, **kw)
    lh, la = op.expected_goals(model, s, fx["home_team"], fx["away_team"], **kw)
    masks = om.market_masks(mg, tl, ml)
    for k, name in enumerate(om.market_names(tl, ml)):
        want = {"home_rate": lh.mean(0), "away_rate": la.mean(0)}.get(name)
        if want is None:
            want = (grid * masks[name]).sum(axis=(1, 2))
        np.testing.assert_allclose(v[:, k], want, rtol=0, atol=1e-15, err_msg=name)


def _hand_fitted(cls, **extra):
    """A predictor whose posterior attributes are set by hand (no fit, no GPU)."""
    p = cls()
    S, T = 8, 3
    s = make_samples(p.model, S, T, 2, seed=3)
    p.teams = ["A", "B", "C"]
    p._teams_dict = {t: i for i, t in enumerate(p.teams)}
    for k, v in s.items():
        setattr(p, k, v)
    for k, v in extra.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("kw,match", [
    (dict(total_lines=(2,)), "half-integer"),
    (dict(total_lines=(2.0,)), "half-integer"),
    (dict(margin_lines=(1,)), "half-integer"),
    (dict(total_lines=(2.25,)), "half-integer"),
    (dict(total_lines=(-0.5,)), "outside"),
    (dict(total_lines=(29.5, 30.5)), "outside"),
    (dict(margin_lines=(-15.5,)), "outside"),
    (dict(margin_lines=(14.5, 15.5)), "outside"),
    (dict(total_lines=tuple(np.arange(17) + 0.5)), "at most 16"),
    (dict(margin_lines=tuple(np.arange(-8, 9) + 0.5)), "at most 16"),
    (dict(total_lines=(2.5, 2.5)), "twice"),
    (dict(quantiles=(0.5, 1.5)), r"\[0, 1\]"),
    (dict(quantiles=(-0.1,)), r"\[0, 1\]"),
    (dict(quantiles=(np.nan,)), r"\[0, 1\]"),
    (dict(quantiles=tuple(np.linspace(0, 1, 9))), "at most 8"),
    (dict(odds={"home_win": 1.0}), "> 1"),
    (dict(odds={"home_win": 0.5}), "> 1"),
    (dict(odds={"draw": np.inf}), "> 1"),
    (dict(odds={"draw": np.nan}), "> 1"),
    (dict(odds={"away_win": [2.0, np.nan]}), "> 1"),
    (dict(odds={"away_win": [2.0, 3.0, 4.0]}), "one value per fixture"),
    (dict(odds={"home_rate": 2.0}), "expected number of goals"),
    (dict(odds={"away_rate": 2.0}), "expected number of goals"),
    (dict(odds={"total_over_9.5": 2.0}), "not a row"),
    (dict(odds={"correct_score_1_0": 7.0}), "not a row"),
    (dict(max_goals=64), r"\[1, 63\]"),
])
def test_refusals_without_a_gpu(kw, match, monkeypatch):
    import torch

    from bpl_next_b200 import DixonColesMatchPredictor

    def no_gpu(*a, **k):
        raise AssertionError("GPU work before the arguments were validated")

    monkeypatch.setattr(torch.Tensor, "cuda", no_gpu)
    p = _hand_fitted(DixonColesMatchPredictor)
    with pytest.raises(ValueError, match=match):
        p.predict_proba_posterior(["A", "B"], ["B", "C"], **kw)


def test_refusals_of_every_class_signature(monkeypatch):
    import torch

    from bpl_next_b200 import (DynamicNeutralDixonColesMatchPredictor, ExtendedDixonColesMatchPredictor,
                               NeutralDixonColesMatchPredictor, NeutralDixonColesMatchPredictorWC)

    monkeypatch.setattr(torch.Tensor, "cuda", lambda *a, **k: (_ for _ in ()).throw(AssertionError("GPU work")))
    with pytest.raises(ValueError, match="half-integer"):
        _hand_fitted(ExtendedDixonColesMatchPredictor).predict_proba_posterior("A", "B", total_lines=(3,))
    with pytest.raises(ValueError, match="half-integer"):
        _hand_fitted(NeutralDixonColesMatchPredictor).predict_proba_posterior("A", "B", 1, margin_lines=(0,))
    wc = _hand_fitted(NeutralDixonColesMatchPredictorWC, _conferences_dict={"X": 0, "Y": 1})
    with pytest.raises(ValueError, match="expected number of goals"):
        wc.predict_proba_posterior("A", "B", "X", "Y", 0, odds={"away_rate": 3.0})
    dyn = DynamicNeutralDixonColesMatchPredictor()
    with pytest.raises(NotImplementedError):
        dyn.predict_proba_posterior("A", "B", 0)
    dyn.teams, dyn._teams_dict = ["A", "B"], {"A": 0, "B": 1}
    dyn.attack, dyn.defence = [np.zeros((4, 2), np.float32)], [np.zeros((4, 2), np.float32)]
    dyn.corr_coef = np.zeros(4, np.float32)
    with pytest.raises(ValueError, match=r"\[0, 1\]"):
        dyn.predict_proba_posterior("A", "B", 0, quantiles=(2.0,), gameweek=3)


def test_lines_struct_and_prototypes_match_the_header():
    text = open(_abi.os.path.join(_abi._HERE, "..", "include", "bplx.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} bplx_market_lines;", text).group(1)
    decl = re.findall(r"^\s*(int32_t|double)\s+(\w+)(\[BPLX_MARKET_MAX_LINES\])?;", re.sub(r"/\*.*?\*/", "", body),
                      re.M)
    assert [(t, n) for t, n, _ in decl] == [("int32_t", "num_total_lines"), ("int32_t", "num_margin_lines"),
                                            ("double", "total_lines"), ("double", "margin_lines")]
    assert [f[0] for f in _abi.MarketLines._fields_] == [n for _, n, _ in decl]
    for name, value in (("BPLX_MARKET_MAX_LINES", _abi.MARKET_MAX_LINES),
                        ("BPLX_QUANTILE_MAX_LEVELS", _abi.QUANTILE_MAX_LEVELS)):
        assert re.search(rf"#define {name} (\d+)", text).group(1) == str(value), name
    assert C.sizeof(_abi.MarketLines) == 8 + 2 * 16 * 8 and _abi.MarketLines.margin_lines.offset == 8 + 16 * 8

    class Stub:  # takes argtypes / restypes of any symbol: no library needed
        def __getattr__(self, name):
            f = type("F", (), {})()
            setattr(self, name, f)
            return f

    lib = _abi.declare(Stub())
    src = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for fn, restype in (("bplx_market_draws_workspace_bytes", C.c_size_t), ("bplx_market_draws", C.c_int),
                        ("bplx_row_quantiles", C.c_int)):
        params = re.search(rf"\b{fn}\(([^;]*)\);", src).group(1)
        assert len(getattr(lib, fn).argtypes) == params.count(",") + 1, fn
        assert getattr(lib, fn).restype == restype, fn
    assert lib.bplx_market_draws.argtypes[3] == C.POINTER(_abi.MarketLines)
    assert lib.bplx_market_draws_workspace_bytes.argtypes[3] == C.POINTER(_abi.MarketLines)


def test_bad_lines_are_refused_by_the_library():
    lib = _abi.lib()
    ln = _abi.MarketLines()
    ln.num_total_lines, ln.total_lines[0] = 1, 2.0  # an integer line
    assert lib.bplx_market_draws_workspace_bytes(None, None, 10, C.byref(ln)) == 0
    assert lib.bplx_row_quantiles(None, 1, 1, 1, None, 0, None, None, None, None) == _abi.E_INVALID
    lv = (C.c_double * 1)(1.5)
    dummy = C.c_void_p(16)
    assert lib.bplx_row_quantiles(dummy, 1, 1, 1, lv, 1, None, dummy, None, None) == _abi.E_INVALID
    assert b"outside [0, 1]" in lib.bplx_last_error()
