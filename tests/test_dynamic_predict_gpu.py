"""GPU: the dynamic model's predictive distribution -- forecast kernel, segmented pointwise log-likelihood, multi-gameweek
posterior predictive check, the predictor API and an end-to-end comparison with a static fit."""
import numpy as np
import pytest
import torch

from bpl_next_b200 import ppc as bppc
from oracle import dynamic_predict as odp
from oracle import predict as op

pytestmark = pytest.mark.gpu


def _dev(d):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in d.items()}


def _gw_samples(G, S, T, seed):
    """NEUTRAL-form samples of G gameweeks ``[G, S, T]`` (corr_coef ``[G, S]``, the same per gameweek)."""
    rng = np.random.default_rng(seed)
    s = {k: rng.normal(0, 0.3, (G, S, T)).astype(np.float32) for k in odp.SITES}
    s["defence"] += np.float32(0.2)
    s["corr_coef"] = np.repeat(rng.uniform(-0.15, 0.05, (1, S)), G, axis=0).astype(np.float32)
    return s


def _slab(s, g):
    return {k: v[g] for k, v in s.items()}


def _matches(sizes, T, seed):
    """Matches grouped by gameweek with ``sizes[g]`` matches at gameweek g, then shuffled."""
    rng = np.random.default_rng(seed)
    gw = np.repeat(np.arange(len(sizes)), sizes)
    M = len(gw)
    h = rng.integers(0, T, M)
    a = (h + rng.integers(1, T, M)) % T
    obs = {"home_team": h.astype(np.uint16), "away_team": a.astype(np.uint16),
           "neutral_venue": (rng.random(M) < 0.25).astype(np.uint8),
           "home_goals": rng.poisson(1.4, M).astype(np.uint8), "away_goals": rng.poisson(1.1, M).astype(np.uint8)}
    perm = rng.permutation(M)
    return {k: v[perm] for k, v in obs.items()}, gw[perm]


# ---- forecast --------------------------------------------------------------------------------------------------------
def test_forecast_replays_the_oracle_and_ignores_draw_ranges():
    """Sites equal the float64 replay on the same words (the device's Box-Muller uses __sincosf: about 1e-6 absolute
    per normal, carried along the walk), and cutting the draws into ranges (a different CTA for every draw) changes no
    bit."""
    from bpl_next_b200 import dynamic_forecast

    S, T, h, seed = 203, 7, 4, 77
    rng = np.random.default_rng(3)
    att, dfn = rng.normal(0, 0.4, (S, T)).astype(np.float32), rng.normal(0, 0.4, (S, T)).astype(np.float32)
    out = dynamic_forecast(torch.from_numpy(att).cuda(), torch.from_numpy(dfn).cuda(), h, seed, first_draw=5)
    ref = odp.forecast(att, dfn, h, seed, first_draw=5)
    for k in odp.SITES:
        np.testing.assert_allclose(out[k].cpu().numpy(), ref[k], rtol=1e-6, atol=2e-5, err_msg=k)
    for cut in (1, 64, 150):
        a = dynamic_forecast(torch.from_numpy(att[:cut]).cuda(), torch.from_numpy(dfn[:cut]).cuda(), h, seed, 5)
        b = dynamic_forecast(torch.from_numpy(att[cut:]).cuda(), torch.from_numpy(dfn[cut:]).cuda(), h, seed, 5 + cut)
        for k in odp.SITES:
            assert torch.equal(torch.cat([a[k], b[k]], dim=1), out[k]), (cut, k)
    # the horizon only appends gameweeks
    longer = dynamic_forecast(torch.from_numpy(att).cuda(), torch.from_numpy(dfn).cuda(), h + 2, seed, 5)
    for k in odp.SITES:
        assert torch.equal(longer[k][:h], out[k])


# ---- segmented pointwise log-likelihood ---------------------------------------------------------------------------------
def test_segmented_pointwise_against_oracle_and_per_gameweek_calls():
    """Ragged gameweeks (0, 1, 257 matches, ...), S = 203 (not a multiple of 4), matches in shuffled order: the matrix
    and statistics equal per-gameweek NEUTRAL calls on the slices bit for bit, and the oracle to float32 rounding."""
    from bpl_next_b200 import pointwise_loglik, pointwise_loglik_gameweeks

    sizes, S, T = [3, 0, 1, 257, 40, 0, 511], 203, 9
    s = _gw_samples(len(sizes), S, T, seed=1)
    obs, gw = _matches(sizes, T, seed=2)
    ll, st = pointwise_loglik_gameweeks("neutral", _dev(s), _dev(obs), gw)
    ll, st = ll.cpu().numpy(), st.cpu().numpy()
    for g in range(len(sizes)):
        m = np.flatnonzero(gw == g)
        if len(m) == 0:
            continue
        ll_g, st_g = pointwise_loglik("neutral", _dev(_slab(s, g)), _dev({k: v[m] for k, v in obs.items()}))
        np.testing.assert_array_equal(ll[m], ll_g.cpu().numpy())
        np.testing.assert_array_equal(st[m], st_g.cpu().numpy())
    want = odp.pointwise_loglik({g: _slab(s, g) for g in range(len(sizes))}, gw, obs["home_team"], obs["away_team"],
                                obs["home_goals"], obs["away_goals"], obs["neutral_venue"])
    got = ll.T.astype(np.float64)
    np.testing.assert_array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    np.testing.assert_allclose(got[fin], want[fin], rtol=1e-5, atol=1e-5)
    # a grouped call writes into a caller's buffer; the statistics do not depend on the matrix
    order = np.argsort(gw, kind="stable")
    buf = torch.full((len(gw), S + 5), np.nan, dtype=torch.float32, device="cuda")
    llb, stb = pointwise_loglik_gameweeks("neutral", _dev(s), _dev({k: v[order] for k, v in obs.items()}), gw[order],
                                          loglik=buf)
    _, st0 = pointwise_loglik_gameweeks("neutral", _dev(s), _dev(obs), gw, want_matrix=False)
    np.testing.assert_array_equal(llb.cpu().numpy(), ll[order])
    assert torch.isnan(buf[:, S:]).all()
    np.testing.assert_array_equal(st0.cpu().numpy(), st)


def test_segmented_calls_refuse_malformed_gameweeks():
    from bpl_next_b200 import _abi
    from bpl_next_b200.problem import _dptr, _gameweek_major, _gw_observations, _samples_struct, _device_ptr_fn
    import ctypes as C

    s = _dev(_gw_samples(3, 16, 5, seed=4))
    obs, gw = _matches([4, 4, 4], 5, seed=5)
    flat, G, S = _gameweek_major(s)
    keep = []
    smp = _samples_struct("neutral", flat, _device_ptr_fn(keep))
    lib = _abi.lib()
    stats = torch.empty((12, 4), dtype=torch.float64, device="cuda")
    # 48 rows are not 5 gameweeks; a gameweek 3 >= G'; not grouped; no gameweek
    for bad, ngw in ((np.sort(gw), 5), (np.sort(gw) + 1, 3), (gw, 3), (np.sort(gw), 0)):
        o, g32 = _gw_observations(flat, _dev(obs), bad, keep)
        ws = torch.empty(1 << 24, dtype=torch.uint8, device="cuda")
        rc = lib.bplx_pointwise_loglik_gameweeks(C.byref(smp), ngw, C.byref(o), g32.ctypes.data, None, 0,
                                                 _dptr(stats), _dptr(ws), ws.numel(), None)
        assert rc == _abi.E_INVALID, (bad, ngw, lib.bplx_last_error())
    assert lib.bplx_pointwise_loglik_gameweeks(C.byref(smp), 3, C.byref(o), None, None, 0, _dptr(stats), _dptr(ws),
                                               ws.numel(), None) == _abi.E_INVALID


# ---- multi-gameweek posterior predictive check -------------------------------------------------------------------------
def test_multi_gameweek_ppc_replays_the_oracle():
    """Scores equal the oracle's replay on the same words except where the oracle's margin is at float32 rounding
    (< 1e-5); the statistics are those of the kernel's own scores; draw ranges give the rows of one call."""
    from bpl_next_b200 import posterior_predictive_gameweeks

    sizes, S, T, R, seed = [30, 0, 57, 14], 61, 8, 2, 31
    s = _gw_samples(len(sizes), S, T, seed=6)
    obs, gw = _matches(sizes, T, seed=7)
    k = posterior_predictive_gameweeks("neutral", _dev(s), _dev(obs), gw, 15, 6, (3, 1), R, seed, want_scores=True)
    k = {n: (None if v is None else v.cpu().numpy()) for n, v in k.items()}
    home, away, margin, valid = odp.replicate({g: _slab(s, g) for g in range(len(sizes))}, gw, obs, 15, R, seed)
    assert k["invalid"][0] == 0 and valid.all()
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    diff = (kh != home) | (ka != away)
    assert not (diff & ~(margin < 1e-5)).any()
    assert diff.sum() <= 1e-3 * diff.size
    st = odp.statistics(obs["home_team"], obs["away_team"], kh, ka, T, 6, (3, 1))
    for name in bppc.STATISTICS:
        np.testing.assert_array_equal(k[name], st[name], err_msg=name)
    lo = posterior_predictive_gameweeks("neutral", _dev({n: v[:, :20] for n, v in s.items()}), _dev(obs), gw, 15, 6,
                                        (3, 1), R, seed, first_draw=0, want_scores=True)
    hi = posterior_predictive_gameweeks("neutral", _dev({n: v[:, 20:] for n, v in s.items()}), _dev(obs), gw, 15, 6,
                                        (3, 1), R, seed, first_draw=20, want_scores=True)
    np.testing.assert_array_equal(np.concatenate([lo["scores"].cpu().numpy(), hi["scores"].cpu().numpy()]),
                                  k["scores"])


def test_one_gameweek_ppc_is_the_neutral_call():
    from bpl_next_b200 import posterior_predictive, posterior_predictive_gameweeks

    S, T, seed = 97, 10, 8
    s = _gw_samples(1, S, T, seed=9)
    obs, gw = _matches([333], T, seed=10)
    a = posterior_predictive_gameweeks("neutral", _dev(s), _dev(obs), gw, 12, 5, (3, 1), 3, seed, first_draw=4,
                                       want_scores=True)
    b = posterior_predictive("neutral", _dev(_slab(s, 0)), _dev(obs), 12, 5, (3, 1), 3, seed, first_draw=4,
                             want_scores=True)
    for name in list(bppc.STATISTICS) + ["scores", "invalid"]:
        assert torch.equal(a[name], b[name]), name


# ---- predictor API -------------------------------------------------------------------------------------------------
def _fake_fit(S=256, T=6, G=3, seed=11):
    """An intended-walk predictor with the attributes ``fit`` records (no sampling)."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor

    rng = np.random.default_rng(seed)
    p = DynamicNeutralDixonColesMatchPredictor()
    p.teams = [f"t{i}" for i in range(T)]
    p._teams_dict = {t: i for i, t in enumerate(p.teams)}
    walk = np.cumsum(rng.normal(0, 0.15, (S, G, T)), axis=1)
    p.attack = [walk[:, g].astype(np.float32) for g in range(G)]
    p.defence = [(0.1 + 0.5 * walk[:, g]).astype(np.float32) for g in range(G)]
    for nm in odp.EFFECTS:
        setattr(p, nm, rng.normal(0.05 if nm.startswith("home") else -0.05, 0.1, (S, G, T)).astype(np.float32))
    p.corr_coef = rng.uniform(-0.1, 0.05, S).astype(np.float32)
    return p


def test_fitted_gameweek_methods_equal_at_gameweek():
    p = _fake_fit()
    h, a, nv = ["t0", "t1", "t2"], ["t3", "t4", "t5"], [0, 1, 0]
    for g in (0, 2):
        q = p.at_gameweek(g)
        np.testing.assert_array_equal(p.predict_score_grid_proba(h, a, nv, gameweek=g)[0],
                                      q.predict_score_grid_proba(h, a, nv)[0])
        po, qo = p.predict_outcome_proba(h, a, nv, knockout=True, gameweek=g), q.predict_outcome_proba(h, a, nv, True)
        for k in qo:
            np.testing.assert_array_equal(po[k], qo[k])
        np.testing.assert_array_equal(p.predict_score_proba(h, a, [1, 0, 2], [1, 1, 0], nv, gameweek=g),
                                      q.predict_score_proba(h, a, [1, 0, 2], [1, 1, 0], nv))
        np.testing.assert_array_equal(p.predict_score_n_proba([0, 2], "t1", "t2", gameweek=g),
                                      q.predict_score_n_proba([0, 2], "t1", "t2"))
        np.testing.assert_array_equal(p.predict_concede_n_proba([1], "t1", "t2", home=False, gameweek=g),
                                      q.predict_concede_n_proba([1], "t1", "t2", home=False))
        for k, v in q.sample_score(h, a, nv, num_samples=50, random_state=3).items():
            np.testing.assert_array_equal(p.sample_score(h, a, nv, 50, random_state=3, gameweek=g)[k], v)
        np.testing.assert_array_equal(p.sample_outcome(h, a, nv, num_samples=40, random_state=4, gameweek=g),
                                      q.sample_outcome(h, a, nv, num_samples=40, random_state=4))
        fx = {"home_team": ["t0", "t1", "t2", "t3"], "away_team": ["t1", "t2", "t3", "t0"]}
        rp, rq = p.simulate_table(fx, random_state=5, gameweek=g), q.simulate_table(fx, random_state=5)
        np.testing.assert_array_equal(rp["position_proba"], rq["position_proba"])
    # the default is the latest fitted gameweek; per-fixture gameweeks are grouped
    np.testing.assert_array_equal(p.predict_score_grid_proba(h, a, nv)[0],
                                  p.predict_score_grid_proba(h, a, nv, gameweek=2)[0])
    mixed = p.predict_score_grid_proba(h, a, nv, gameweek=[0, 2, 0])[0]
    np.testing.assert_array_equal(mixed[[0, 2]], p.predict_score_grid_proba(h, a, nv, gameweek=0)[0][[0, 2]])
    np.testing.assert_array_equal(mixed[1], p.predict_score_grid_proba(h, a, nv, gameweek=2)[0][1])


def test_forecast_gameweek_methods_equal_the_oracle():
    p = _fake_fit()
    G = len(p.attack)
    h, a, nv = np.array([0, 1, 2]), np.array([3, 4, 5]), np.array([0, 1, 0])
    for g in (G, G + 3):
        grid, _, _ = p.predict_score_grid_proba(h, a, nv, max_goals=8, gameweek=g, random_state=21)
        fc = odp.forecast(p.attack[-1], p.defence[-1], g - G + 1, 21)
        smp = {k: v[g - G] for k, v in fc.items()}
        smp["corr_coef"] = p.corr_coef
        want, _, _ = op.predict_score_grid_proba("neutral", smp, h, a, 8, neutral_venue=nv)
        np.testing.assert_allclose(grid, want, rtol=0, atol=1e-6)
        again, _, _ = p.predict_score_grid_proba(h, a, nv, max_goals=8, gameweek=g, random_state=21)
        np.testing.assert_array_equal(grid, again)
    other, _, _ = p.predict_score_grid_proba(h, a, nv, max_goals=8, gameweek=G, random_state=22)
    assert not np.array_equal(other, p.predict_score_grid_proba(h, a, nv, max_goals=8, gameweek=G, random_state=21)[0])


def test_pointwise_matches_predict_score_proba_and_loo_runs():
    """exp(ll) averaged over the draws is predict_score_proba at each match's gameweek (fitted and forecast)."""
    p = _fake_fit()
    rng = np.random.default_rng(12)
    M = 60
    h = rng.integers(0, 6, M)
    a = (h + rng.integers(1, 6, M)) % 6
    data = {"home_team": [p.teams[i] for i in h], "away_team": [p.teams[i] for i in a],
            "home_goals": rng.poisson(1.3, M), "away_goals": rng.poisson(1.1, M),
            "neutral_venue": (rng.random(M) < 0.2).astype(int), "gameweek": rng.integers(0, 5, M)}
    ll = p.log_likelihood(data, random_state=9)  # [S, M]
    want = np.empty(M)
    for g in np.unique(data["gameweek"]):
        m = np.flatnonzero(data["gameweek"] == g)
        want[m] = p.predict_score_proba(h[m], a[m], data["home_goals"][m], data["away_goals"][m],
                                        data["neutral_venue"][m], gameweek=int(g), random_state=9)
    np.testing.assert_allclose(np.exp(ll.astype(np.float64)).mean(axis=0), want, rtol=0, atol=1e-6)
    ls = p.log_score(data, random_state=9)
    np.testing.assert_allclose(np.exp(ls["pointwise"]), want, rtol=0, atol=1e-6)
    # (forecast gameweeks have HalfNormal(1) spreads: some draws put tau below 0, so ll = -inf there and p_waic is
    # undefined; lppd, the log of the averaged probability, stays finite and is the log score)
    w = p.waic(data, random_state=9)
    assert w["num_matches"] == M
    np.testing.assert_allclose(w["lppd"], ls["log_score"], rtol=1e-12)


# ---- end to end ------------------------------------------------------------------------------------------------------
def _drifting_league(seed=3, T=8, G=6):
    """Two legs per gameweek; attack strengths swing by about 1.5 over six gameweeks (strong drift)."""
    rng = np.random.default_rng(seed)
    names = [f"club{i}" for i in range(T)]
    base = np.linspace(-1.0, 1.0, T)
    ht, at, hg, ag, gw = [], [], [], [], []
    for g in range(G):
        att = base * np.cos(np.pi * g / (G - 1))  # the order of the table reverses from gameweek 0 to G - 1
        for i in range(T):
            for j in range(T):
                if i != j:
                    ht.append(names[i]); at.append(names[j]); gw.append(g)
                    hg.append(rng.poisson(np.exp(0.1 + att[i] - 0.0)))
                    ag.append(rng.poisson(np.exp(-0.1 + att[j] - 0.0)))
    return {"home_team": ht, "away_team": at, "home_goals": np.array(hg), "away_goals": np.array(ag),
            "gameweek": np.array(gw), "neutral_venue": np.zeros(len(ht), np.int64),
            "game_weights": np.ones(len(ht)), "time_diff": np.zeros(len(ht))}


def test_end_to_end_dynamic_beats_static_on_a_drifting_league():
    """A league whose attack strengths reverse over six gameweeks.  The static NEUTRAL fit averages the strengths away;
    the walk follows them.  compare() ranks the dynamic fit first on the training data by a wide margin (the data
    give about 3 log-points per team-gameweek of swing; the test asks for 20 elpd over 336 matches), and its posterior
    predictive check finds no team's points out of line (p-values in [0.01, 0.99])."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor, NeutralDixonColesMatchPredictor
    from bpl_next_b200.compare import compare

    td = _drifting_league()
    kw = dict(num_warmup=300, num_samples=200, mcmc_kwargs={"num_chains": 16})
    dyn = DynamicNeutralDixonColesMatchPredictor().fit(td, random_state=1, **kw)
    sta = NeutralDixonColesMatchPredictor().fit(td, random_state=1, **kw)
    res = compare({"dynamic": dyn.loo(), "static": sta.loo()})
    assert res["dynamic"]["rank"] == 0, res
    print("E2E", {k: (v["elpd_loo"], v["d_elpd"], v["dse"], v["p_loo"]) for k, v in res.items()})
    chk = dyn.posterior_predictive_check(random_state=2)
    p = chk["team_points"]["p_value"]
    chk_s = sta.posterior_predictive_check(random_state=2)
    print("E2E pvals dyn", np.round(p, 3), "static", np.round(chk_s["team_points"]["p_value"], 3))
    assert (p > 0.01).all() and (p < 0.99).all(), p
    # the last gameweek's table order is the reverse of the first's
    g0 = dyn.predict_outcome_proba("club7", "club0", 0, gameweek=0)["home_win"][0]
    g5 = dyn.predict_outcome_proba("club7", "club0", 0, gameweek=5)["home_win"][0]
    assert g5 < 0.5 < g0
