"""CPU checks of the model-comparison oracle (oracle/psis.py) and of the host arithmetic of bpl_next_b200.compare."""
import numpy as np
import pytest
import torch
from scipy.special import logsumexp
from scipy.stats import norm

from oracle import models as om, psis


def gpd_draws(rng, k, n, sigma=1.0):
    u = rng.random(n)
    return sigma * np.expm1(-k * np.log1p(-u)) / k


@pytest.mark.parametrize("k", [0.2, 0.5, 0.9])
def test_gpd_shape_is_recovered(k):
    """Importance ratios drawn from a generalised Pareto distribution: the mean k-hat over 20 replicates of 4,000 draws
    is within three standard errors of the true shape."""
    rng = np.random.default_rng(11)
    ks = np.array([psis.psislw(np.log(gpd_draws(rng, k, 4000)))[1] for _ in range(20)])
    assert np.isfinite(ks).all()
    se = ks.std(ddof=1) / np.sqrt(len(ks))
    assert abs(ks.mean() - k) < 3 * se, (ks.mean(), se)


def test_psis_loo_matches_exact_loo_on_a_conjugate_normal_model():
    """y_i ~ N(mu, 1), mu ~ N(0, 10^2), n = 50, S = 4,000 exact posterior draws: PSIS-LOO is within 0.01 of the exact
    leave-one-out predictive density, and every k-hat is below 0.5."""
    rng = np.random.default_rng(3)
    n, S, tau2 = 50, 4000, 100.0
    y = rng.normal(0.7, 1.0, n)

    def posterior(yy):
        v = 1.0 / (1.0 / tau2 + len(yy))
        return v * yy.sum(), v

    m, v = posterior(y)
    mu = rng.normal(m, np.sqrt(v), S)
    ll = norm.logpdf(y[None, :], loc=mu[:, None], scale=1.0)
    exact = 0.0
    for i in range(n):
        mi, vi = posterior(np.delete(y, i))
        exact += norm.logpdf(y[i], loc=mi, scale=np.sqrt(1.0 + vi))
    res = psis.loo(ll)
    assert abs(res["elpd_loo"] - exact) < 0.01, (res["elpd_loo"], exact)
    assert (res["pareto_k"] < 0.5).all()


def test_psis_edge_cases():
    """S = 1 and a tail of at most 4 draws give k-hat = inf and no smoothing; a non-finite entry gives (NaN, inf); tied
    draws give the same result in any order."""
    e, k = psis.loo_pointwise(np.array([[-1.5]]))
    assert k[0] == np.inf and e[0] == pytest.approx(-1.5, abs=1e-15)
    rng = np.random.default_rng(0)
    ll = rng.normal(-2, 0.3, (20, 3))  # Mt = 4: the tail has at most 4 draws
    e, k = psis.loo_pointwise(ll)
    assert np.isinf(k).all()
    np.testing.assert_allclose(e, np.log(20) - logsumexp(-ll, axis=0), rtol=1e-12)  # raw importance weights
    ll[5, 1] = -np.inf
    e, k = psis.loo_pointwise(ll)
    assert np.isnan(e[1]) and k[1] == np.inf and np.isfinite(e[[0, 2]]).all()
    col = np.repeat(rng.normal(-2, 0.5, 250), 4)
    e1, k1 = psis.loo_pointwise(col[:, None])
    e2, k2 = psis.loo_pointwise(rng.permutation(col)[:, None])
    assert e1[0] == pytest.approx(e2[0], rel=1e-13) and k1[0] == pytest.approx(k2[0], rel=1e-12)


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
def test_oracle_loglik_sums_to_the_model_likelihood(model):
    """sum_m of the pointwise log-likelihood equals the likelihood part of oracle/models.py (unweighted data), for the
    corr_coef the model derives from its bounds."""
    rng = np.random.default_rng(5)
    S, T, Cf, M = 6, 7, 3, 60
    h = rng.integers(0, T, M)
    a = (h + rng.integers(1, T, M)) % T
    d = om.MatchData(model=model, num_teams=T, home_team=h, away_team=a, home_goals=rng.poisson(1.4, M),
                     away_goals=rng.poisson(1.1, M))
    t = {"attack": rng.normal(0, 0.3, (S, T)), "defence": rng.normal(0, 0.3, (S, T)),
         "corr_coef_raw": rng.uniform(0.2, 0.8, S)}
    fx = {}
    if model == "dixon_coles":
        t["home_advantage"] = rng.normal(0.25, 0.1, S)
    elif model == "extended":
        t["home_advantage"] = rng.normal(0.25, 0.1, (S, T))
    else:
        for k in ("home_attack", "away_attack", "home_defence", "away_defence"):
            t[k] = rng.normal(0, 0.1, (S, T))
        d.neutral_venue = (rng.random(M) < 0.4).astype(np.int64)
        fx["neutral_venue"] = d.neutral_venue
        if model == "neutral_wc":
            t["confederation_strength"] = rng.normal(0, 0.2, (S, Cf))
            d.home_conf, d.away_conf, d.num_conferences = rng.integers(0, Cf, M), rng.integers(0, Cf, M), Cf
            fx["home_conf"], fx["away_conf"] = d.home_conf, d.away_conf
    total, cc = om.likelihood_from_tables(d, {k: torch.as_tensor(v, dtype=torch.float64) for k, v in t.items()})
    samples = {k: v for k, v in t.items() if k != "corr_coef_raw"}
    samples["corr_coef"] = cc.numpy()
    ll = psis.pointwise_loglik(model, samples, h, a, d.home_goals, d.away_goals, **fx)
    assert ll.shape == (S, M)
    np.testing.assert_allclose(ll.sum(axis=1), total.numpy(), rtol=1e-13)


def test_compare_arithmetic():
    from bpl_next_b200 import compare as bc

    rng = np.random.default_rng(2)
    M, S = 200, 1000
    base = rng.normal(-1.5, 0.4, M)
    res = {}
    for name, shift in (("a", 0.0), ("b", -0.02), ("c", 0.01)):
        e = base + shift + rng.normal(0, 0.05, M)
        lppd = e + 0.01
        k = np.where(np.arange(M) < 3, 0.75, 0.2)
        res[name] = bc.loo_from_pointwise(e, k, lppd, S, match_key="same")
    r = res["a"]
    assert r["elpd_loo"] == pytest.approx(r["pointwise"].sum())
    assert r["se"] == pytest.approx(np.sqrt(M * r["pointwise"].var()))
    assert r["p_loo"] == pytest.approx(0.01 * M)
    assert r["good_k"] == pytest.approx(min(1 - 1 / np.log10(S), 0.7)) and r["n_k_above_0.7"] == 3
    out = bc.compare(res)
    assert list(out) == ["c", "a", "b"]
    best = res["c"]["pointwise"]
    for name, row in out.items():
        diff = best - res[name]["pointwise"]
        assert row["d_elpd"] == pytest.approx(diff.sum()) and row["dse"] == pytest.approx(np.sqrt(M * diff.var()))
        assert set(row) == {"rank", "elpd_loo", "p_loo", "se", "d_elpd", "dse", "n_k_above_0.7"}
    assert out["c"]["d_elpd"] == 0 and out["c"]["dse"] == 0 and out["c"]["rank"] == 0
    res["b"] = dict(res["b"], match_key="other")
    with pytest.raises(ValueError, match="different matches"):
        bc.compare(res)

    stats = np.stack([np.full(M, -1.0), np.full(M, 2.0), np.full(M, -1.0 * S), np.full(M, 1.0 * S + 0.5 * S)], axis=1)
    w = bc.waic_from_stats(stats, S)
    np.testing.assert_allclose(w["lppd_pointwise"], -1.0 + np.log(2.0) - np.log(S))
    np.testing.assert_allclose(w["p_waic_pointwise"], 0.5)
    assert w["elpd_waic"] == pytest.approx(M * (-1.0 + np.log(2.0) - np.log(S) - 0.5))


def test_waic_oracle_matches_definitions():
    rng = np.random.default_rng(4)
    ll = rng.normal(-2, 0.5, (300, 12))
    w = psis.waic(ll)
    lppd = np.log(np.exp(ll).mean(axis=0))
    np.testing.assert_allclose(w["pointwise"], lppd - ll.var(axis=0), rtol=1e-12)
