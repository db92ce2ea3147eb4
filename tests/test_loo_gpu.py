"""GPU parity of model comparison: the pointwise log-likelihood kernel and the PSIS-LOO kernel against the float64
oracle (oracle/psis.py), against K1's likelihood entry point and predict_score_proba, and the predictor methods end to
end."""
import numpy as np
import pytest
import torch

from bpl_next_b200 import data as bdata
from oracle import datasets, psis
from tests.test_score_grid_gpu import make_fixtures, make_samples

pytestmark = pytest.mark.gpu


def _goals(M, seed):
    """Poisson(1.3) scores with 0-0, 1-0, 0-1, 1-1 and scores of 9 and more among the first matches."""
    rng = np.random.default_rng(seed)
    hg, ag = rng.poisson(1.3, M), rng.poisson(1.1, M)
    fixed = [(0, 0), (1, 0), (0, 1), (1, 1), (9, 2), (3, 11), (10, 10)]
    for i, (h, a) in enumerate(fixed[:M]):
        hg[i], ag[i] = h, a
    return hg.astype(np.uint8), ag.astype(np.uint8)


def _to_dev(d):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in d.items()}


def _oracle_ll(model, s, fx, hg, ag):
    kw = {k: fx[k] for k in ("home_conf", "away_conf", "neutral_venue") if k in fx}
    return psis.pointwise_loglik(model, s, fx["home_team"], fx["away_team"], hg, ag, **kw)


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("S,M,pad", [(1, 37, 3), (3, 5000, 1), (203, 300, 5), (4097, 1, 7), (4097, 300, 3)])
def test_pointwise_against_oracle(model, S, M, pad):
    """ll of every (draw, match) within |d| <= 2e-5 + 2e-6 |ll| of the float64 oracle: the kernel works in float32 --
    rates are products of float32 exponentials (a few ulp, ~5e-7 relative), and y log(rate) with scores up to 11 turns
    that into up to ~1e-5 absolute; the Poisson and tau terms then add float32 rounding proportional to |ll|.
    The statistics are those of the kernel's own matrix (sums in float64), and a call without the matrix returns the
    same statistics bit for bit.  ld = S + pad > S."""
    from bpl_next_b200 import pointwise_loglik

    T, Cf = 9, 4
    s = make_samples(model, S, T, Cf, seed=S + 1)
    fx = make_fixtures(model, M, T, Cf, seed=M + 2)
    hg, ag = _goals(M, seed=3)
    obs = dict(fx, home_goals=hg, away_goals=ag)
    buf = torch.full((M, S + pad), np.nan, dtype=torch.float32, device="cuda")
    ll, st = pointwise_loglik(model, _to_dev(s), _to_dev(obs), loglik=buf)
    _, st0 = pointwise_loglik(model, _to_dev(s), _to_dev(obs), want_matrix=False)
    torch.cuda.synchronize()
    assert torch.equal(st, st0)
    assert torch.isnan(buf[:, S:]).all()  # nothing written past S
    got = ll.cpu().numpy().T.astype(np.float64)  # [S, M]
    want = _oracle_ll(model, s, fx, hg, ag)
    # (draws with corr_coef beyond the bounds of a match's rates have tau < 0 on a low-score cell: -inf in both)
    np.testing.assert_array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert fin.all() or S > 1000
    err = np.abs(got[fin] - want[fin])
    assert (err <= 2e-5 + 2e-6 * np.abs(want[fin])).all(), err.max()
    st = st.cpu().numpy()
    from scipy.special import logsumexp
    np.testing.assert_array_equal(st[:, 0], got.max(axis=0))
    np.testing.assert_allclose(st[:, 0] + np.log(st[:, 1]), logsumexp(got, axis=0), rtol=0, atol=1e-6)
    np.testing.assert_allclose(st[:, 2], got.sum(axis=0), rtol=1e-12)
    np.testing.assert_allclose(st[:, 3], (got ** 2).sum(axis=0), rtol=1e-12)


def test_pointwise_tau_clamped_and_errors():
    """A corr_coef far outside its bounds makes tau <= 0 on 0-0 and 1-1: ll = -inf there, as in predict; DYNAMIC, ld < S and
    missing goals are refused."""
    from bpl_next_b200 import _abi, pointwise_loglik

    S, T, M = 16, 5, 8
    s = make_samples("dixon_coles", S, T, 0, seed=3)
    s["corr_coef"] = np.full(S, 5.0, dtype=np.float32)
    fx = make_fixtures("dixon_coles", M, T, 0, seed=4)
    hg, ag = _goals(M, seed=1)
    ll, _ = pointwise_loglik("dixon_coles", _to_dev(s), _to_dev(dict(fx, home_goals=hg, away_goals=ag)))
    ll = ll.cpu().numpy()
    assert np.isneginf(ll[0]).all() and np.isneginf(ll[3]).all() and np.isfinite(ll[4:7]).all()
    with pytest.raises(_abi.BplxError):
        pointwise_loglik("dynamic", _to_dev(s), _to_dev(dict(fx, home_goals=hg, away_goals=ag)))
    with pytest.raises(_abi.BplxError):
        pointwise_loglik("dixon_coles", _to_dev(s), _to_dev(dict(fx, home_goals=hg, away_goals=ag)),
                         loglik=torch.empty((M, S), device="cuda")[:, :S - 1].contiguous())


@pytest.mark.parametrize("model,make", [("dixon_coles", datasets.dummy_data), ("neutral", datasets.neutral_dummy_data),
                                        ("neutral_wc", datasets.neutral_dummy_data)])
def test_sum_over_matches_equals_the_likelihood_entry_point(model, make):
    """On unweighted data, sum_m ll[s, m] equals K1's likelihood entry point (Problem.loglik) for the same draws and the
    corr_coef it returns.  K1 sums M float32 terms, so the tolerance is that of a float32 sum (rtol 1e-5)."""
    from bpl_next_b200 import Problem, pointwise_loglik

    arr, _ = bdata.prepare(model, make())
    arr.weights = None
    p = Problem(arr)
    lay = p.loglik_layout
    Dl = sum(c for _, c, _ in lay.values())
    C = 64
    rng = np.random.default_rng(12)
    tabs = rng.normal(0, 0.3, (C, Dl)).astype(np.float32)
    tabs[:, lay["corr_coef_raw"][0]] = rng.uniform(0.05, 0.95, C)
    ll_k1, _, cc = p.loglik(torch.from_numpy(tabs).cuda())
    s = {name: np.ascontiguousarray(tabs[:, off:off + cnt]) for name, (off, cnt, _) in lay.items()
         if name != "corr_coef_raw"}
    if model == "dixon_coles":
        s["home_advantage"] = np.ascontiguousarray(s["home_advantage"][:, 0])
    s["corr_coef"] = cc.cpu().numpy()
    obs = {"home_team": arr.home_team, "away_team": arr.away_team, "home_goals": arr.home_goals,
           "away_goals": arr.away_goals}
    for k in ("neutral_venue", "home_conf", "away_conf"):
        if getattr(arr, k) is not None:
            obs[k] = getattr(arr, k).astype(np.uint8)
    ll, _ = pointwise_loglik(model, _to_dev(s), _to_dev(obs))
    total = ll.cpu().numpy().astype(np.float64).sum(axis=0)
    np.testing.assert_allclose(total, ll_k1.cpu().numpy(), rtol=1e-5)


def test_log_score_equals_predict_score_proba():
    """exp of the held-out pointwise log score is predict_score_proba of those matches (NeutralWC, with conferences and
    neutral venues) to 1e-6."""
    from bpl_next_b200 import NeutralDixonColesMatchPredictorWC

    td = datasets.neutral_dummy_data()
    n = len(td["home_team"])
    idx_train, idx_test = np.arange(0, n - 90), np.arange(n - 90, n)

    def take(ix):
        return {k: ([v[i] for i in ix] if isinstance(v, list) else np.asarray(v)[ix]) for k, v in td.items()}

    m = NeutralDixonColesMatchPredictorWC().fit(take(idx_train), num_warmup=150, num_samples=100,
                                               mcmc_kwargs={"num_chains": 8})
    test = take(idx_test)
    res = m.log_score(test)
    p = m.predict_score_proba(test["home_team"], test["away_team"], test["home_conf"], test["away_conf"],
                              test["home_goals"], test["away_goals"], test["neutral_venue"])
    assert res["num_matches"] == 90 and res["log_score"] == pytest.approx(res["pointwise"].sum())
    np.testing.assert_allclose(np.exp(res["pointwise"]), p, rtol=0, atol=1e-6)


def _psis_rows(S, seed):
    """Rows: light tails, heavy tails (k-hat > 0.7), repeated draws (ties), the same ties in another order, a -inf."""
    rng = np.random.default_rng(seed)
    rows = [rng.normal(-2.0, 0.3, S)]
    u = rng.random(S)
    rows.append(-np.log(np.expm1(-1.0 * np.log1p(-u)) / 1.0 + 1e-3) - 1.0)  # ratios ~ GPD(k = 1)
    tied = np.round(rng.normal(-1.5, 0.5, S), 1)
    rows += [tied, rng.permutation(tied)]
    bad = rng.normal(-2.0, 0.3, S)
    bad[S // 2] = -np.inf
    rows.append(bad)
    return np.stack(rows).astype(np.float32)  # [M, S]


@pytest.mark.parametrize("S", [1, 20, 100, 4000, 100_000])
@pytest.mark.parametrize("r_eff", [1.0, 0.3])
def test_psis_against_oracle(S, r_eff):
    """The PSIS kernel and the oracle on the same float32 matrix: k-hat to 1e-6, elpd_loo_m to 1e-9 relative.  Rows
    longer than shared memory (S = 100,000), tails of at most 4 draws (S <= 20: k-hat = inf), heavy tails, ties (two
    orders of the same tied draws give the same k-hat bits) and a non-finite entry (NaN, inf)."""
    from bpl_next_b200 import psis_loo

    X = _psis_rows(S, seed=S)
    buf = torch.zeros((X.shape[0], S + 3), dtype=torch.float32, device="cuda")
    buf[:, :S] = torch.from_numpy(X).cuda()
    e, k = psis_loo(buf[:, :S], r_eff)
    e, k = e.cpu().numpy(), k.cpu().numpy()
    e_o, k_o = psis.loo_pointwise(X.T.astype(np.float64), r_eff)
    assert np.isnan(e[4]) and k[4] == np.inf and np.isnan(e_o[4])
    fin = slice(0, 4)
    np.testing.assert_allclose(e[fin], e_o[fin], rtol=1e-9)
    np.testing.assert_array_equal(np.isinf(k[fin]), np.isinf(k_o[fin]))
    np.testing.assert_allclose(k[fin][np.isfinite(k_o[fin])], k_o[fin][np.isfinite(k_o[fin])], rtol=0, atol=1e-6)
    # the tail is sorted, so k-hat is the same bits; the body is summed in row order, so elpd may differ by rounding
    assert k[2] == k[3] and e[2] == pytest.approx(e[3], rel=1e-13)
    if S <= 20:
        assert np.isinf(k[fin]).all()
    if S >= 4000:
        assert k_o[1] > 0.7


def test_psis_long_rows_and_limits():
    """S = 2^24 draws per row (Mt = 12,288); a tail above the 16,384-draw limit and r_eff <= 0 are refused."""
    from bpl_next_b200 import _abi, psis_loo

    S = 1 << 24
    rng = np.random.default_rng(8)
    x = rng.normal(-2.0, 0.4, S).astype(np.float32)
    e, k = psis_loo(torch.from_numpy(x).cuda()[None, :])
    e_o, k_o = psis.loo_pointwise(x[:, None].astype(np.float64))
    np.testing.assert_allclose(e.cpu().numpy(), e_o, rtol=1e-9)
    np.testing.assert_allclose(k.cpu().numpy(), k_o, rtol=0, atol=1e-6)
    with pytest.raises(_abi.BplxError, match="16384"):
        psis_loo(torch.zeros((1, 1 << 22), device="cuda"), r_eff=0.01)
    with pytest.raises(_abi.BplxError):
        psis_loo(torch.zeros((2, 10), device="cuda"), r_eff=0.0)


@pytest.fixture(scope="module")
def dc_fit():
    from bpl_next_b200 import DixonColesMatchPredictor

    return DixonColesMatchPredictor().fit(datasets.dummy_data(), num_warmup=300, num_samples=500,
                                          mcmc_kwargs={"num_chains": 8})


def test_loo_is_deterministic_and_independent_of_match_ranges(dc_fit, monkeypatch):
    from bpl_next_b200 import predictors

    a, b = dc_fit.loo(), dc_fit.loo()
    monkeypatch.setattr(predictors, "LOO_MATRIX_BYTES", 4 * 4000 * 37)  # ranges of 37 matches
    c = dc_fit.loo()
    for r in (b, c):
        assert np.array_equal(a["pointwise"], r["pointwise"]) and np.array_equal(a["pareto_k"], r["pareto_k"])
        assert a["elpd_loo"] == r["elpd_loo"] and a["p_loo"] == r["p_loo"]


def test_end_to_end_against_the_oracle(dc_fit):
    """loo() and waic() of a DixonColes fit of the reference's dummy_data (8 chains) equal the oracle run on the
    predictor's own log_likelihood() matrix; compare() of that fit and an Extended fit gives the documented keys; the
    dynamic class raises."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor, ExtendedDixonColesMatchPredictor
    from bpl_next_b200.compare import compare

    ll = dc_fit.log_likelihood()
    assert ll.shape == (4000, 380) and ll.dtype == np.float32
    lo, lw = dc_fit.loo(), dc_fit.waic()
    o_lo, o_w = psis.loo(ll), psis.waic(ll)
    np.testing.assert_allclose(lo["pointwise"], o_lo["pointwise"], rtol=1e-9)
    np.testing.assert_allclose(lo["pareto_k"], o_lo["pareto_k"], rtol=0, atol=1e-6)
    assert lo["elpd_loo"] == pytest.approx(o_lo["elpd_loo"], rel=1e-9)
    assert lo["se"] == pytest.approx(o_lo["se"], rel=1e-6)
    # lppd comes from the pointwise kernel's sum of float32 exponentials: ~1e-7 per match
    assert lo["p_loo"] == pytest.approx(o_lo["p_loo"], abs=380 * 2e-7)
    assert lo["n_k_above_0.7"] == o_lo["n_k_above_0.7"]
    np.testing.assert_allclose(lw["pointwise"], o_w["pointwise"], rtol=0, atol=1e-6)
    assert lw["elpd_waic"] == pytest.approx(o_w["elpd_waic"], abs=380 * 1e-6)
    assert lw["p_waic"] == pytest.approx(o_w["p_waic"], rel=1e-6)

    ext = ExtendedDixonColesMatchPredictor().fit(datasets.dummy_data(), num_warmup=300, num_samples=500,
                                                 mcmc_kwargs={"num_chains": 8})
    out = compare({"dc": lo, "ext": ext.loo()})
    assert sorted(out) == ["dc", "ext"]
    for row in out.values():
        assert set(row) == {"rank", "elpd_loo", "p_loo", "se", "d_elpd", "dse", "n_k_above_0.7"}
    best = min(out, key=lambda n: out[n]["rank"])
    assert out[best]["d_elpd"] == 0.0 and all(r["d_elpd"] >= 0 for r in out.values())

    dyn = DynamicNeutralDixonColesMatchPredictor()
    for call in (dyn.loo, dyn.waic, dyn.log_likelihood):
        with pytest.raises(NotImplementedError):
            call()
    with pytest.raises(NotImplementedError):
        dyn.log_score(datasets.dummy_data())
