"""CPU: the dynamic model's predictive distribution -- fitted-gameweek rates pinned to the likelihood, the forecast's
word map and distributions, the C prototypes, and the predictor's refusals."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch
from scipy import stats

from bpl_next_b200 import _abi
from oracle import dynamic_predict as odp
from oracle import models as om
from oracle import philox
from oracle import predict as op

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _small_case(seed=0):
    """6 teams (team 5 plays no match), 4 gameweeks, covariates, some neutral venues."""
    rng = np.random.default_rng(seed)
    T, G, M = 6, 4, 40
    home = rng.integers(0, 5, M)
    away = (home + rng.integers(1, 5, M)) % 5
    d = om.MatchData(model="dynamic", num_teams=T, home_team=home, away_team=away,
                     home_goals=rng.integers(0, 5, M), away_goals=rng.integers(0, 5, M),
                     neutral_venue=(rng.random(M) < 0.3).astype(np.int64), covariates=rng.normal(size=(T, 2)),
                     gameweek=rng.integers(0, G, M), num_gameweeks=G, walk="intended")
    return d


def test_fitted_gameweek_rates_equal_the_likelihood():
    d = _small_case()
    D = om.num_params("dynamic", d.num_teams, 2, 0, d.num_gameweeks)
    theta = np.random.default_rng(1).uniform(-1.5, 1.5, (16, D))
    _, det = om.log_density(d, torch.as_tensor(theta, dtype=torch.float64))
    lam_h, lam_a = det["lam_h"].numpy(), det["lam_a"].numpy()
    sites = odp.fitted_sites(theta, d.num_teams, d.num_gameweeks, d.covariates)
    cc = det["corr_coef"].numpy()
    for m in range(d.num_matches):
        sl = odp.slab(sites, int(d.gameweek[m]), cc)
        lh, la = op.expected_goals("neutral", sl, d.home_team[m:m + 1], d.away_team[m:m + 1],
                                   neutral_venue=d.neutral_venue[m:m + 1])
        np.testing.assert_allclose(lh[:, 0], lam_h[:, m], rtol=1e-12, atol=0)
        np.testing.assert_allclose(la[:, 0], lam_a[:, m], rtol=1e-12, atol=0)


def test_forecast_words_by_hand():
    seed, T, h, first = 12345, 3, 2, 7
    w = odp.forecast_words(seed, T, h, first, 2)
    key = seed ^ 0x9E3779B97F4A7C15
    P = 3 + 3 * T
    for s in range(2):
        for k in range(h):
            for b in range(P):
                assert tuple(int(x) for x in w[s, k, b]) == philox.block(key, first + s, k * P + b)
    # draw 1, gameweek 1, team 2, by hand from its words
    att0 = np.array([[0.3, -0.2, 0.1], [0.5, 0.0, -0.4]])
    def0 = np.array([[0.1, 0.2, 0.3], [-0.1, 0.4, 0.0]])
    fc = odp.forecast(att0, def0, h, seed, first)
    s, t = 1, 2
    att, dfn = att0[s, t], def0[s, t]
    for k in range(h):
        bd = [philox.block(key, first + s, k * P + b) for b in range(3)]
        bt = [philox.block(key, first + s, k * P + 3 + 3 * t + b) for b in range(3)]
        words = [x for blk in bt for x in blk]
        u = sorted(float(philox.uniform(x)) for x in words[:5])[1]
        rho = 2.0 * u - 1.0
        za, eps = philox.box_muller(words[6], words[7])
        zd = rho * za + np.sqrt(1.0 - rho * rho) * eps
        std_a, std_d = (abs(v) for v in philox.box_muller(bd[2][0], bd[2][1]))
        att, dfn = att + za * std_a, dfn + zd * std_d
        m_ha = 0.1 + 0.2 * philox.box_muller(bd[0][0], bd[0][1])[0]
        s_ha = abs(philox.box_muller(bd[1][0], bd[1][1])[0])
        dec_ha = philox.box_muller(words[8], words[9])[0]
        m_ad = -0.1 + 0.2 * philox.box_muller(bd[0][2], bd[0][3])[1]
        s_ad = abs(philox.box_muller(bd[1][2], bd[1][3])[1])
        dec_ad = philox.box_muller(words[10], words[11])[1]
        assert fc["attack"][k, s, t] == pytest.approx(att, abs=1e-13)
        assert fc["defence"][k, s, t] == pytest.approx(dfn, abs=1e-13)
        assert fc["home_attack"][k, s, t] == pytest.approx(m_ha + s_ha * dec_ha, abs=1e-13)
        assert fc["away_defence"][k, s, t] == pytest.approx(m_ad + s_ad * dec_ad, abs=1e-13)


def test_forecast_distributions():
    n = 100_000
    v = odp.forecast_variates(odp.forecast_words(2024, 1, 1, 0, n))
    u = v["u"][:, 0, 0]
    assert stats.kstest(u, stats.beta(2, 4).cdf).pvalue > 1e-4

    def within(x, mean):
        x = np.asarray(x, np.float64).ravel()
        assert abs(x.mean() - mean) < 5 * x.std() / np.sqrt(len(x)), (x.mean(), mean)

    for k in ("std_attack", "std_defence", "std_home_attack", "std_away_defence"):
        within(v[k], np.sqrt(2 / np.pi))
    within(v["mean_home_attack"], 0.1)
    within(v["mean_away_defence"], -0.1)
    za, eps = v["za"][:, 0, 0], v["eps"][:, 0, 0]
    rho = 2.0 * u - 1.0
    zd = rho * za + np.sqrt(1.0 - rho ** 2) * eps
    within(za * zd, -1.0 / 3.0)  # corr(za, zd) = E[rho] (unit variances)
    inc = za * v["std_attack"][:, 0]  # one step of the attack walk
    within(inc, 0.0)
    within(inc ** 2, 1.0)


def _prototypes():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bplx.h")).read(), flags=re.S)
    out = {}
    for m in re.finditer(r"(size_t|int)\s+(bplx_[a-z_0-9]+)\(([^;]*?)\);", src, flags=re.S):
        out[m.group(2)] = (m.group(1), [a for a in m.group(3).split(",") if a.strip()])
    return out


@pytest.mark.parametrize("name", ["bplx_dynamic_forecast", "bplx_pointwise_loglik_gameweeks_workspace_bytes",
                                  "bplx_pointwise_loglik_gameweeks",
                                  "bplx_posterior_predictive_gameweeks_workspace_bytes",
                                  "bplx_posterior_predictive_gameweeks"])
def test_prototypes_match_header(name):
    ret, args = _prototypes()[name]
    fn = getattr(_abi.lib(), name)
    assert len(fn.argtypes) == len(args), (name, args)
    assert fn.restype == (C.c_size_t if ret == "size_t" else C.c_int)
    src = open(os.path.join(ROOT, "include", "bplx.h")).read()
    assert re.search(r"#define BPLX_FORECAST_KEY 0x%Xull" % _abi.FORECAST_KEY, src)
    assert re.search(r"#define BPLX_FORECAST_MAX_TEAMS %d\b" % _abi.FORECAST_MAX_TEAMS, src)


def test_gameweek_calls_refuse_without_touching_the_gpu():
    lib = _abi.lib()
    assert lib.bplx_pointwise_loglik_gameweeks_workspace_bytes(None, 1, None) == 0
    assert lib.bplx_posterior_predictive_gameweeks_workspace_bytes(None, 1, None) == 0
    assert lib.bplx_dynamic_forecast(None, None, 4, 3, 1, 0, 0, *([None] * 6), None) == _abi.E_INVALID
    buf = (C.c_float * 12)()
    p = C.cast(buf, C.c_void_p)
    assert lib.bplx_dynamic_forecast(p, p, 4, 3, 0, 0, 0, *([p] * 6), None) == _abi.E_INVALID  # horizon < 1
    assert b"horizon" in lib.bplx_last_error()
    assert lib.bplx_dynamic_forecast(p, p, 4, 300, 1, 0, 0, *([p] * 6), None) == _abi.E_UNSUPPORTED


def _fake_fit(walk):
    """A dynamic predictor with the attributes ``fit`` records (no sampling): 8 draws, 3 teams, 2 gameweeks."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor

    rng = np.random.default_rng(0)
    S, T, G = 8, 3, 2
    p = DynamicNeutralDixonColesMatchPredictor(walk=walk)
    p.teams, p._teams_dict = ["a", "b", "c"], {"a": 0, "b": 1, "c": 2}
    p.attack = [rng.normal(size=(S, T)).astype(np.float32) for _ in range(G)]
    p.defence = [rng.normal(size=(S, T)).astype(np.float32) for _ in range(G)]
    for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
        setattr(p, nm, rng.normal(size=(S, G, T)).astype(np.float32))
    p.corr_coef = rng.uniform(-0.1, 0.1, S).astype(np.float32)
    return p


def _predictive_calls(p):
    return [
        lambda: p.at_gameweek(0),
        lambda: p.predict_score_grid_proba("a", "b", 0),
        lambda: p.predict_outcome_proba("a", "b", 0),
        lambda: p.predict_score_proba("a", "b", 1, 0, 0),
        lambda: p.predict_score_n_proba(1, "a", "b"),
        lambda: p.predict_concede_n_proba(1, "a", "b"),
        lambda: p.sample_score("a", "b", 0),
        lambda: p.sample_outcome("a", "b", 0),
        lambda: p.simulate_table({"home_team": ["a"], "away_team": ["b"]}),
        lambda: p.simulate_tournament(None, []),
        lambda: p.log_likelihood(),
        lambda: p.waic(),
        lambda: p.loo(),
        lambda: p.log_score({"home_team": ["a"], "away_team": ["b"], "home_goals": [1], "away_goals": [0],
                             "neutral_venue": [0], "gameweek": [0]}),
        lambda: p.posterior_predictive_check(),
    ]


def test_predictive_methods_need_an_intended_walk_fit():
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor

    for p in (DynamicNeutralDixonColesMatchPredictor(), DynamicNeutralDixonColesMatchPredictor(walk="as_written"),
              _fake_fit("as_written")):
        for call in _predictive_calls(p):
            with pytest.raises(NotImplementedError, match='walk="intended"'):
                call()


def test_negative_gameweek_is_refused():
    p = _fake_fit("intended")
    for call in (lambda: p.at_gameweek(-1), lambda: p.predict_score_grid_proba("a", "b", 0, gameweek=-2),
                 lambda: p.predict_outcome_proba(["a", "b"], ["b", "c"], 0, gameweek=[0, -1]),
                 lambda: p.simulate_table({"home_team": ["a"], "away_team": ["b"]}, gameweek=-1)):
        with pytest.raises(ValueError, match="gameweek"):
            call()
