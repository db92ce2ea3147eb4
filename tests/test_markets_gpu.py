"""GPU: per-draw market probabilities (bplx_market_draws) against the float64 oracle, their statistics and exact
quantiles (bplx_row_quantiles) against numpy on the kernel's own matrix, and predict_proba_posterior end to end."""
import numpy as np
import pytest
import torch

from bpl_next_b200 import predictors as bp
from bpl_next_b200.problem import market_draws, market_names, row_quantiles, score_grid
from oracle import markets as om
from tests.test_dynamic_predict_gpu import _fake_fit
from tests.test_score_grid_gpu import make_fixtures, make_samples

pytestmark = pytest.mark.gpu
LINES = {4: ((0.5, 2.5, 7.5), (-3.5, -0.5, 0.5, 3.5)),
         15: ((1.5, 2.5, 3.5, 29.5), (-14.5, -1.5, 1.5)),
         40: ((0.5, 4.5, 79.5), (-39.5, 2.5))}
LEVELS = (0.0, 0.05, 0.25, 0.5, 0.75, 0.95, 1.0, 1.0 / 3.0)


def _dev(d):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in d.items()}


def _fx_kw(fx):
    return {k: fx[k] for k in ("home_conf", "away_conf", "neutral_venue") if k in fx}


def _sd(x):
    """sd (divisor S) along the last axis of float32 values, from their exact differences to the first value."""
    d = x.astype(np.float64) - x[..., :1].astype(np.float64)
    return np.sqrt(((d - d.mean(-1, keepdims=True)) ** 2).mean(-1))


def _edges(x, odds):
    return ((x.astype(np.float64) * odds[:, None]) > 1.0).sum(-1)


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("G", [4, 15, 40])
def test_draws_against_the_oracle_and_statistics_against_numpy(model, G):
    S, F, T, Cf = 149, 301, 7, 4
    s = make_samples(model, S, T, Cf, seed=21)
    fx = make_fixtures(model, F, T, Cf, seed=22)
    tl, ml = LINES[G]
    names = market_names(tl, ml)
    K = len(names)
    mat, st, inv = market_draws(model, _dev(s), _dev(fx), G, tl, ml)
    torch.cuda.synchronize()
    assert int(inv.item()) == 0
    m = mat.cpu().numpy()
    ref = om.market_draws(model, s, fx["home_team"], fx["away_team"], G, tl, ml, **_fx_kw(fx))  # [S, F, K]
    ref = ref.transpose(1, 2, 0).reshape(F * K, S)
    rate = np.isin(np.tile(names, F), ["home_rate", "away_rate"])
    np.testing.assert_allclose(m[~rate], ref[~rate], rtol=0, atol=1e-5)
    np.testing.assert_allclose(m[rate], ref[rate], rtol=2e-6, atol=0)
    st = st.cpu().numpy()
    np.testing.assert_allclose(st[:, 0], m.astype(np.float64).mean(-1), rtol=1e-12, atol=0)
    np.testing.assert_allclose(st[:, 1], _sd(m), rtol=1e-12, atol=0)
    # the same statistics without the matrix
    _, st2, _ = market_draws(model, _dev(s), _dev(fx), G, tl, ml, want_matrix=False)
    np.testing.assert_array_equal(st2.cpu().numpy(), st)
    # quantiles and edge counts, exactly numpy's
    rng = np.random.default_rng(G)
    odds = np.where(rng.random(F * K) < 0.2, 0.0, rng.uniform(1.01, 12.0, F * K))
    q, e = row_quantiles(mat, LEVELS, torch.from_numpy(odds).cuda())
    np.testing.assert_array_equal(q.cpu().numpy(), np.quantile(m.astype(np.float64), LEVELS, axis=-1).T)
    np.testing.assert_array_equal(e.cpu().numpy(), _edges(m, odds))


@pytest.mark.parametrize("model,G", [("dixon_coles", 15), ("neutral_wc", 10), ("extended", 40)])
def test_means_are_the_averaged_grid(model, G):
    S, F, T, Cf = 203, 97, 9, 3
    s = make_samples(model, S, T, Cf, seed=5)
    fx = make_fixtures(model, F, T, Cf, seed=6)
    tl, ml = LINES[15] if G < 29 else LINES[40]
    tl, ml = tuple(x for x in tl if x < 2 * G), tuple(x for x in ml if abs(x) < G)
    names = market_names(tl, ml)
    _, st, _ = market_draws(model, _dev(s), _dev(fx), G, tl, ml, want_matrix=False)
    grid, outcome = score_grid(model, _dev(s), _dev(fx), G)
    mean = st.cpu().numpy()[:, 0].reshape(F, len(names))
    g = grid.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(mean[:, :3], outcome.cpu().numpy(), rtol=0, atol=1e-6)
    masks = om.market_masks(G, tl, ml)
    for k, name in enumerate(names):
        if name in masks:
            np.testing.assert_allclose(mean[:, k], (g * masks[name]).sum(axis=(1, 2)), rtol=0, atol=1e-6, err_msg=name)


def _hand_fitted(cls, S, T, seed, **extra):
    p = cls()
    p.teams = [f"t{i}" for i in range(T)]
    p._teams_dict = {t: i for i, t in enumerate(p.teams)}
    for k, v in make_samples(p.model, S, T, 3, seed=seed).items():
        setattr(p, k, v)
    for k, v in extra.items():
        setattr(p, k, v)
    return p


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], dict):
            _assert_same(a[k], b[k])
        elif isinstance(a[k], np.ndarray):
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        else:
            assert a[k] == b[k], k


def test_ranges_and_batches_change_no_bit(monkeypatch):
    from bpl_next_b200 import NeutralDixonColesMatchPredictor

    S, T, F = 300, 8, 50
    p = _hand_fitted(NeutralDixonColesMatchPredictor, S, T, seed=9)
    rng = np.random.default_rng(4)
    h = rng.integers(0, T, F)
    a = (h + rng.integers(1, T, F)) % T
    home, away, nv = [p.teams[i] for i in h], [p.teams[i] for i in a], list(rng.integers(0, 2, F))
    odds = {"home_win": rng.uniform(1.5, 4.0, F), "total_over_2.5": 1.9}
    full = p.predict_proba_posterior(home, away, nv, odds=odds, return_draws=True)
    K = len(full["markets"])
    monkeypatch.setattr(bp, "MARKET_MATRIX_BYTES", 4 * S * K * 3)  # ranges of 3 fixtures
    _assert_same(p.predict_proba_posterior(home, away, nv, odds=odds, return_draws=True), full)
    monkeypatch.undo()
    one = p.predict_proba_posterior(home[17], away[17], nv[17], odds={"home_win": odds["home_win"][17],
                                                                       "total_over_2.5": 1.9}, return_draws=True)
    sub = {k: ({kk: vv[17:18] for kk, vv in v.items()} if isinstance(v, dict) else v) for k, v in full.items()}
    sub["draws"] = full["draws"][17:18]
    _assert_same(one, sub)


@pytest.mark.parametrize("S", [1, 2, 3, 1000, 1 << 22])
def test_row_quantiles_are_numpys(S):
    rng = np.random.default_rng(S)
    R = 7 if S < (1 << 20) else 3
    rows = np.empty((R, S), np.float32)
    rows[0] = rng.random(S)                                              # spread
    rows[1] = np.float32(0.3125)                                         # constant
    rows[2] = rng.choice(np.float32([0.0, 0.25, 0.5, 0.75, 1.0]), S)     # heavy ties, zeros
    if R > 3:
        rows[3] = rng.choice(np.float32([0.0, 1e-45, 3e-42, 1e-39, 1.1754942e-38, 2e-38]), S)  # zeros and denormals
        rows[4] = rng.normal(0, 1, S).astype(np.float32)                     # negative values
        rows[5] = np.float32(0.5) + rng.integers(0, 3, S).astype(np.float32) * np.float32(2 ** -23)  # adjacent floats
        rows[6] = (rng.random(S) ** 8).astype(np.float32)                    # crowded near 0
    pad = torch.zeros((R, S + 5), dtype=torch.float32, device="cuda")   # a row pitch larger than S
    pad[:, :S] = torch.from_numpy(rows).cuda()
    odds = np.linspace(0.0, 6.0, R)
    q, e = row_quantiles(pad[:, :S], LEVELS, torch.from_numpy(odds).cuda())
    np.testing.assert_array_equal(q.cpu().numpy(), np.quantile(rows.astype(np.float64), LEVELS, axis=-1).T)
    np.testing.assert_array_equal(e.cpu().numpy(), _edges(rows, odds))
    q3, e3 = row_quantiles(pad[:, :S], (0.5,))
    assert e3 is None
    np.testing.assert_array_equal(q3.cpu().numpy()[:, 0], np.quantile(rows.astype(np.float64), 0.5, axis=-1))


def test_a_non_finite_rate_raises():
    from bpl_next_b200 import DixonColesMatchPredictor

    p = _hand_fitted(DixonColesMatchPredictor, 64, 4, seed=2)
    p.attack = p.attack.copy()
    p.attack[10, 1] = np.inf
    s = {k: getattr(p, k) for k in ("attack", "defence", "home_advantage", "corr_coef")}
    fx = {"home_team": np.array([1, 0, 2], np.uint16), "away_team": np.array([0, 1, 3], np.uint16)}
    _, _, inv = market_draws("dixon_coles", _dev(s), _dev(fx), 10, (2.5,), ())
    assert int(inv.item()) == 2  # draw 10 of the two fixtures of team 1
    with pytest.raises(ValueError, match="non-finite"):
        p.predict_proba_posterior(["t1", "t2"], ["t0", "t3"])


def _check_end_to_end(res, outcome, S, lv=(0.05, 0.5, 0.95)):
    assert res["num_draws"] == S and list(res["quantile_levels"]) == list(lv)
    d = res["draws"]
    for k, name in enumerate(res["markets"]):
        r = res[name]
        np.testing.assert_allclose(r["mean"], d[:, k].astype(np.float64).mean(-1), rtol=1e-12, atol=0)
        np.testing.assert_array_equal(r["quantiles"], np.quantile(d[:, k].astype(np.float64), lv, axis=-1).T)
    for k, name in enumerate(("home_win", "draw", "away_win")):
        np.testing.assert_allclose(res[name]["mean"], outcome[name], rtol=0, atol=1e-6)


def test_end_to_end_on_every_class():
    from bpl_next_b200 import (DixonColesMatchPredictor, ExtendedDixonColesMatchPredictor,
                               NeutralDixonColesMatchPredictor, NeutralDixonColesMatchPredictorWC)

    S, T = 500, 6
    home, away = ["t0", "t1", "t2", "t5"], ["t3", "t4", "t5", "t0"]
    for cls in (DixonColesMatchPredictor, ExtendedDixonColesMatchPredictor):
        p = _hand_fitted(cls, S, T, seed=1)
        res = p.predict_proba_posterior(home, away, odds={"draw": 3.4}, return_draws=True)
        _check_end_to_end(res, p.predict_outcome_proba(home, away), S)
        assert np.array_equal(res["draw"]["edge_proba"], _edges(res["draws"][:, 1], np.full(4, 3.4)) / S)
        np.testing.assert_allclose(res["draw"]["expected_value"], res["draw"]["mean"] * 3.4 - 1.0, rtol=1e-15)
    p = _hand_fitted(NeutralDixonColesMatchPredictor, S, T, seed=2)
    nv = [0, 1, 0, 1]
    _check_end_to_end(p.predict_proba_posterior(home, away, nv, return_draws=True),
                      p.predict_outcome_proba(home, away, nv), S)
    p = _hand_fitted(NeutralDixonColesMatchPredictorWC, S, T, seed=3, _conferences_dict={"X": 0, "Y": 1, "Z": 2})
    hc, ac = ["X", "Y", "Z", "X"], ["Z", "Z", "X", "Y"]
    _check_end_to_end(p.predict_proba_posterior(home, away, hc, ac, nv, quantiles=(0.1, 0.9), return_draws=True),
                      p.predict_outcome_proba(home, away, hc, ac, nv), S, (0.1, 0.9))


def test_dynamic_fitted_and_forecast_gameweeks_equal_at_gameweek():
    p = _fake_fit()
    G = len(p.attack)
    h, a, nv = ["t0", "t1", "t2", "t3"], ["t3", "t4", "t5", "t0"], [0, 1, 0, 0]
    gws = [1, G + 1, 1, G - 1]
    odds = {"away_win": [2.5, 3.0, 4.0, 5.0]}
    res = p.predict_proba_posterior(h, a, nv, odds=odds, return_draws=True, gameweek=gws, random_state=7)
    for g in sorted(set(gws)):
        idx = [i for i, x in enumerate(gws) if x == g]
        q = p.at_gameweek(g, random_state=7).predict_proba_posterior(
            [h[i] for i in idx], [a[i] for i in idx], [nv[i] for i in idx],
            odds={"away_win": [odds["away_win"][i] for i in idx]}, return_draws=True)
        for name in res["markets"]:
            for k, v in q[name].items():
                np.testing.assert_array_equal(res[name][k][idx], v, err_msg=(g, name, k))
        np.testing.assert_array_equal(res["draws"][idx], q["draws"])
    out = p.predict_outcome_proba(h, a, nv, gameweek=gws, random_state=7)
    _check_end_to_end(res, out, len(p.corr_coef))
