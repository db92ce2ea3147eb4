"""Posterior predictive checks on the GPU: the kernel replayed exactly by the float64 oracle (oracle/ppc.py) on the same
Philox words, its scores equal to simulate_table's, invariance to draw ranges and seeds, agreement with the predict
path, and the predictor method end to end."""
import ctypes as C

import numpy as np
import pytest
import torch

from bpl_next_b200 import _abi, season
from bpl_next_b200 import ppc as bppc
from oracle import datasets
from oracle import ppc as oppc
from tests.test_score_grid_gpu import make_fixtures, make_samples

pytestmark = pytest.mark.gpu


def _dev(d):
    return {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda()) for k, v in d.items()}


def _obs(model, M, T, Cf, seed):
    """M observed matches between T teams (neutral venues and confederations mixed in) with Poisson scores."""
    fx = make_fixtures(model, M, T, Cf, seed)
    rng = np.random.default_rng(seed + 7)
    return dict(fx, home_goals=rng.poisson(1.4, M).astype(np.uint8), away_goals=rng.poisson(1.1, M).astype(np.uint8))


def _run(model, s, obs, G=15, R=1, seed=1, first_draw=0, B=6, points=(3, 1), scores=True):
    from bpl_next_b200 import posterior_predictive

    out = posterior_predictive(model, _dev(s), _dev(obs), G, B, points, R, seed, first_draw=first_draw,
                               want_scores=scores)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("R,G", [(1, 15), (7, 4), (1, 4), (7, 15)])
def test_exact_replay(model, R, G):
    """Every kernel score equals the oracle's on the same Philox words, except (replicate, match) pairs whose oracle
    margin is below 1e-5 (float32 rounding at a cumulative boundary), at most 0.1 % of them; every statistic equals,
    integer for integer, the oracle's statistics of the kernel's own scores.  S = 149 draws, M = 301 (an odd match
    count: the last Philox block is half used)."""
    S, M, T, Cf, seed = 149, 301, 11, 4, 500 + 10 * R + G
    s = make_samples(model, S, T, Cf, seed=seed)
    obs = _obs(model, M, T, Cf, seed)
    k = _run(model, s, obs, G, R, seed)
    o = oppc.replicate(model, s, obs, G, R, seed)
    home, away, margin, valid = o
    assert k["invalid"][0] == 0 and valid.all()
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    assert kh.max() <= G and ka.max() <= G
    diff = (kh != home) | (ka != away)
    assert not (diff & ~(margin < 1e-5)).any(), np.argwhere(diff & ~(margin < 1e-5))[:5]
    assert diff.sum() <= 1e-3 * diff.size
    st = oppc.statistics(obs["home_team"], obs["away_team"], kh, ka, T, 6, (3, 1))
    for name in bppc.STATISTICS:
        np.testing.assert_array_equal(k[name], st[name], err_msg=name)


def test_score_bins_and_points():
    """Other bins and points: the statistics still equal the oracle's of the kernel's own scores."""
    s = make_samples("neutral_wc", 30, 9, 3, seed=2)
    obs = _obs("neutral_wc", 120, 9, 3, seed=3)
    for B, pts in ((2, (2, 1)), (16, (1, 0))):
        k = _run("neutral_wc", s, obs, 15, 3, seed=4, B=B, points=pts)
        st = oppc.statistics(obs["home_team"], obs["away_team"], k["scores"][:, :, 0], k["scores"][:, :, 1], 9, B, pts)
        for name in bppc.STATISTICS:
            np.testing.assert_array_equal(k[name], st[name], err_msg=name)


def test_equal_to_simulation():
    """A 20-team league: the replicated scores are bit-equal to simulate_table's raw scores with the same seed, draws
    and the matches as fixtures (NeutralWC with neutral venues and confederations, R = 3)."""
    from bpl_next_b200 import simulate_table

    T, Cf, S, R, M = 20, 4, 37, 3, 190
    s = make_samples("neutral_wc", S, T, Cf, seed=11)
    obs = _obs("neutral_wc", M, T, Cf, seed=12)
    names = [f"S{i}" for i in range(T)]
    tab = season.build_table(names)
    hs, as_ = season.fixture_slots(tab, [names[i] for i in obs["home_team"]], [names[i] for i in obs["away_team"]])
    dtab = _dev({k: tab[k] for k in ("start_points", "start_goals_for", "start_goals_against", "group")})
    dtab.update({k: tab[k] for k in ("num_positions", "num_points_bins", "points_win", "points_draw")})
    fx = {k: obs[k] for k in ("home_team", "away_team", "home_conf", "away_conf", "neutral_venue")}
    sim = simulate_table("neutral_wc", _dev(s), _dev(dict(fx, home_slot=hs, away_slot=as_)), dtab, 15, R, 77,
                         want_scores=True)
    k = _run("neutral_wc", s, obs, 15, R, 77)
    np.testing.assert_array_equal(k["scores"], sim["scores"].cpu().numpy())


def test_draw_ranges_and_seeds():
    """Draws [0, 17) and [17, 50) with first_draw: every row equals the single call's; the same seed repeats, another
    seed differs; the statistics do not depend on whether the raw scores are written."""
    s = make_samples("extended", 50, 10, 0, seed=21)
    obs = _obs("extended", 200, 10, 0, seed=22)
    full = _run("extended", s, obs, 15, 3, seed=99)
    parts = [_run("extended", {k: v[lo:hi] for k, v in s.items()}, obs, 15, 3, seed=99, first_draw=lo)
             for lo, hi in ((0, 17), (17, 50))]
    for key in bppc.STATISTICS + ("scores",):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]), err_msg=key)
    again = _run("extended", s, obs, 15, 3, seed=99)
    noraw = _run("extended", s, obs, 15, 3, seed=99, scores=False)
    for key in bppc.STATISTICS:
        np.testing.assert_array_equal(full[key], again[key])
        np.testing.assert_array_equal(full[key], noraw[key])
    assert noraw["scores"] is None
    other = _run("extended", s, obs, 15, 3, seed=100)
    assert not np.array_equal(full["scores"], other["scores"])


def test_against_the_predict_path():
    """N = 2^16 replicates of 40 matches: the replicate mean of score_counts is within 5 Monte-Carlo standard errors
    of the sum over matches of bplx_score_grid's grid (lumped at B - 1), and outcome_counts of the sum of its outcome
    probabilities (the same draws)."""
    from bpl_next_b200 import score_grid

    S, R, M, T, Cf = 64, 1024, 40, 8, 3
    s = make_samples("neutral_wc", S, T, Cf, seed=31)
    obs = _obs("neutral_wc", M, T, Cf, seed=32)
    k = _run("neutral_wc", s, obs, 15, R, seed=5, scores=False)
    fx = {k_: obs[k_] for k_ in ("home_team", "away_team", "home_conf", "away_conf", "neutral_venue")}
    grid, outcome = score_grid("neutral_wc", _dev(s), _dev(fx), 15)
    g = grid.double().cpu().numpy().sum(axis=0)  # [16, 16]
    lumped = np.zeros((6, 6))
    for i in range(16):
        for j in range(16):
            lumped[min(i, 5), min(j, 5)] += g[i, j]
    N = S * R
    for name, want in (("score_counts", lumped), ("outcome_counts", outcome.double().cpu().numpy().sum(axis=0))):
        rep = k[name].astype(np.float64)
        se = rep.std(axis=0) / np.sqrt(N)
        assert (np.abs(rep.mean(axis=0) - want) <= 5 * se + 1e-9).all(), (rep.mean(axis=0) - want) / se


def _raw_call(s, obs, G=15, B=6, pw=3, pd=1, R=1, goals=True):
    """bplx_posterior_predictive called directly (no Python-side checks); returns the status."""
    from bpl_next_b200 import problem

    lib = _abi.lib()
    keep = []
    ptr = problem._device_ptr_fn(keep)
    ds = _dev(s)
    st = problem._samples_struct("dixon_coles", ds, ptr)
    o = _abi.Observations()
    o.fixtures = problem._fixtures_struct(_dev(obs), ptr)
    if goals:
        o.home_goals, o.away_goals = ptr(_dev(obs)["home_goals"]), ptr(_dev(obs)["away_goals"])
    buf = torch.zeros(1 << 20, dtype=torch.int64, device="cuda")
    out = _abi.PpcOutput(*([ptr(buf)] * 7 + [None, ptr(buf)]))
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    rc = lib.bplx_posterior_predictive(C.byref(st), C.byref(o), G, B, pw, pd, R, 1, 0, C.byref(out), ptr(ws),
                                       ws.numel(), None)
    torch.cuda.synchronize()
    return rc


def test_invalid_draws_and_refusals():
    s = make_samples("dixon_coles", 12, 6, 0, seed=41)
    obs = _obs("dixon_coles", 30, 6, 0, seed=42)
    # non-finite rates: those draws' replicates are invalid, their rows -1, the others untouched
    bad = {k: v.copy() for k, v in s.items()}
    bad["attack"][3, obs["home_team"][0]] = np.inf
    bad["defence"][7, obs["away_team"][2]] = np.nan
    k = _run("dixon_coles", bad, obs, 15, 5, seed=4)
    good = _run("dixon_coles", s, obs, 15, 5, seed=4)
    assert k["invalid"][0] == 10
    rows = np.repeat(np.isin(np.arange(12), [3, 7]), 5)
    assert (k["team_points"][rows] == -1).all() and (k["score_counts"][rows] == -1).all()
    assert (k["total_goals_sq"][rows] == -1).all() and (k["goals"][rows] == -1).all()
    np.testing.assert_array_equal(k["team_points"][~rows], good["team_points"][~rows])
    assert (k["scores"][rows] == 255).any(axis=(1, 2)).all()

    # refusals: DYNAMIC, max_goals, score_bins, R, points, missing goals, N >= 2^31
    with pytest.raises(_abi.BplxError):
        _run("dynamic", s, obs)
    for kw in ({"G": 0}, {"G": 64}, {"B": 1}, {"B": 17}, {"R": 0}, {"points": (0, 0)}, {"points": (1, 3)},
               {"points": (3, -1)}):
        with pytest.raises(_abi.BplxError):
            _run("dixon_coles", s, obs, **kw)
    assert _raw_call(s, obs) == _abi.OK
    assert _raw_call(s, obs, goals=False) == _abi.E_INVALID
    assert _raw_call(s, obs, R=(1 << 31) // 12 + 1) == _abi.E_UNSUPPORTED
    assert _raw_call(s, obs, pw=(1 << 31) // 30 + 1, pd=0) == _abi.E_INVALID


def _take(td, ix):
    return {k: ([v[i] for i in ix] if isinstance(v, list) else np.asarray(v)[ix]) for k, v in td.items()}


@pytest.fixture(scope="module")
def dc_fit():
    from bpl_next_b200 import DixonColesMatchPredictor

    return DixonColesMatchPredictor().fit(datasets.dummy_data(), num_warmup=300, num_samples=500,
                                          mcmc_kwargs={"num_chains": 8})


def test_end_to_end(dc_fit, monkeypatch):
    """A DixonColes fit of dummy_data (8 chains): the documented keys and shapes, observed values equal to a direct
    count of the data, a fixed random_state repeats, ranges of draws change nothing, the raw replicates give the
    statistics, and the dynamic class raises."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor, predictors

    td = datasets.dummy_data()
    res = dc_fit.posterior_predictive_check(random_state=3)
    S, T, M = dc_fit.attack.shape[0], len(dc_fit.teams), len(td["home_team"])
    assert res["num_replicates"] == S and res["sims_per_draw"] == 1 and res["seed"] == 3
    assert res["score_bins"] == 6 and res["max_goals"] == predictors.MAX_GOALS and res["teams"] == list(dc_fit.teams)
    assert res["match_key"] == dc_fit.waic()["match_key"]
    shapes = {"score_counts": (6, 6), "outcome_counts": (3,), "goals": (2,), "total_goals_sq": (),
              "team_points": (T,), "team_goals_for": (T,), "team_goals_against": (T,), "total_goals_dispersion": ()}
    for name, shp in shapes.items():
        for field in ("observed", "mean", "sd", "p_value"):
            assert np.shape(res[name][field]) == shp, (name, field)
        assert ((res[name]["p_value"] >= 0) & (res[name]["p_value"] <= 1)).all()
    idx = {t: i for i, t in enumerate(dc_fit.teams)}
    hg, ag = np.asarray(td["home_goals"], np.int64), np.asarray(td["away_goals"], np.int64)
    assert res["goals"]["observed"].tolist() == [hg.sum(), ag.sum()]
    assert res["outcome_counts"]["observed"].tolist() == [(hg > ag).sum(), (hg == ag).sum(), (hg < ag).sum()]
    assert res["score_counts"]["observed"].sum() == M and res["score_counts"]["observed"][1, 1] == ((hg == 1) & (ag == 1)).sum()
    pts = np.zeros(T, np.int64)
    for h, a, x, y in zip(td["home_team"], td["away_team"], hg, ag):
        pts[idx[h]] += 3 if x > y else 1 if x == y else 0
        pts[idx[a]] += 3 if y > x else 1 if x == y else 0
    np.testing.assert_array_equal(res["team_points"]["observed"], pts)

    again = dc_fit.posterior_predictive_check(random_state=3)
    monkeypatch.setattr(predictors, "SIM_OUTPUT_BYTES", 333 * (4 * (36 + 3 + 3 * T) + 24 + 2 * M))  # 333 draws
    raw = dc_fit.posterior_predictive_check(random_state=3, return_replicates=True)
    for r in (again, raw):
        for name in shapes:
            for field in ("observed", "mean", "sd", "p_value"):
                np.testing.assert_array_equal(res[name][field], r[name][field], err_msg=(name, field))
    assert raw["home_score"].shape == (M, S) and raw["away_score"].shape == (M, S)
    st = bppc.statistics([idx[t] for t in td["home_team"]], [idx[t] for t in td["away_team"]], raw["home_score"][:, 5],
                         raw["away_score"][:, 5], T)
    for name in bppc.STATISTICS:
        np.testing.assert_array_equal(raw["replicates"][name][5], st[name])
    other = dc_fit.posterior_predictive_check(random_state=4)
    assert not np.array_equal(other["team_points"]["mean"], res["team_points"]["mean"])

    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().posterior_predictive_check()


def _with_scores(td, hg, ag):
    return dict(td, home_goals=np.asarray(hg, np.int64), away_goals=np.asarray(ag, np.int64))


def test_dispersion_in_and_out_of_the_model():
    """Data drawn from the model (independent Poisson goals of fixed team strengths on dummy_data's fixtures) give a
    dispersion p-value inside (0.05, 0.95).  Negative-binomial goals (variance = mean + mean^2) are over-dispersed: the
    observed dispersion lies above what every replicate shows, so p = P(T_rep > T_obs) + 1/2 P(T_rep = T_obs) is below
    0.01 (the model misses, in the tail of too little spread)."""
    from bpl_next_b200 import DixonColesMatchPredictor

    td = datasets.dummy_data()
    teams = sorted(set(td["home_team"]) | set(td["away_team"]))
    rng = np.random.default_rng(17)
    att, dfn = rng.normal(0, 0.3, len(teams)), rng.normal(0, 0.2, len(teams))
    i = {t: k for k, t in enumerate(teams)}
    h = np.array([i[t] for t in td["home_team"]])
    a = np.array([i[t] for t in td["away_team"]])
    mu_h, mu_a = np.exp(0.25 + att[h] - dfn[a]), np.exp(att[a] - dfn[h])
    fits = {}
    for name, (hg, ag) in {"poisson": (rng.poisson(mu_h), rng.poisson(mu_a)),
                           "negbin": (rng.negative_binomial(1.0, 1.0 / (1.0 + mu_h)),
                                      rng.negative_binomial(1.0, 1.0 / (1.0 + mu_a)))}.items():
        data = _with_scores(td, np.minimum(hg, 20), np.minimum(ag, 20))
        m = DixonColesMatchPredictor().fit(data, num_warmup=300, num_samples=250, mcmc_kwargs={"num_chains": 8})
        fits[name] = m.posterior_predictive_check(random_state=1)["total_goals_dispersion"]
    assert 0.05 < fits["poisson"]["p_value"] < 0.95, fits["poisson"]
    neg = fits["negbin"]
    assert neg["p_value"] < 0.01 and neg["observed"] > neg["mean"] + 5 * neg["sd"], neg


def test_invalid_draws_raise_through_the_predictor():
    from bpl_next_b200 import DixonColesMatchPredictor

    s = make_samples("dixon_coles", 12, 6, 0, seed=51)
    s["attack"][4, 1] = np.inf
    m = DixonColesMatchPredictor()
    m.teams = np.array([f"T{i}" for i in range(6)])
    m._teams_dict = {t: i for i, t in enumerate(m.teams)}
    m.attack, m.defence, m.home_advantage, m.corr_coef = s["attack"], s["defence"], s["home_advantage"], s["corr_coef"]
    data = {"home_team": ["T1", "T2", "T3"], "away_team": ["T0", "T1", "T5"], "home_goals": [1, 0, 2],
            "away_goals": [0, 0, 1]}
    with pytest.raises(ValueError, match="non-finite"):
        m.posterior_predictive_check(data, random_state=1)
    with pytest.raises(ValueError, match="1 of 12 replicates"):  # one draw, one replicate per draw
        m.posterior_predictive_check(dict(data, home_team=["T2", "T2", "T1"], away_team=["T0", "T4", "T5"]),
                                     random_state=1)
    res = m.posterior_predictive_check(dict(data, home_team=["T2", "T2", "T3"], away_team=["T0", "T4", "T5"]),
                                       random_state=1)  # T1 plays in no match: every draw is usable
    assert res["num_replicates"] == 12
