"""Season / group-stage simulation on the GPU: the kernel replayed exactly by the float64 oracle (oracle/simulate.py) on
the same Philox words, draw-range invariance, agreement with the predict path, tau clamp / invalid draws / refusals, and
the predictor method end to end."""
import ctypes as C

import numpy as np
import pytest
import torch

from bpl_next_b200 import _abi, season
from oracle import datasets
from oracle import predict as op
from oracle import simulate as osim
from tests.test_score_grid_gpu import make_samples

pytestmark = pytest.mark.gpu


def _dev(d):
    return {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda()) for k, v in d.items()}


def _dev_table(tab):
    d = _dev({k: tab[k] for k in ("start_points", "start_goals_for", "start_goals_against", "group")})
    d.update({k: tab[k] for k in ("num_positions", "num_points_bins", "points_win", "points_draw")})
    return d


def _case(model, S, T_tab, grouped, F, seed, Cf=4):
    """Samples for T_tab + 3 model teams, a table of T_tab slots mapped to a random subset of them (with a random start),
    F random fixtures between slots (neutral venues mixed, random confederations)."""
    T = T_tab + 3
    s = make_samples(model, S, T, Cf, seed=seed)
    rng = np.random.default_rng(seed + 1)
    team_of_slot = rng.permutation(T)[:T_tab]
    names = [f"S{i}" for i in range(T_tab)]
    groups = None
    if grouped:
        groups = [f"g{(i * 7) % 5}" for i in range(T_tab)] if T_tab > 20 else [f"g{i // 4}" for i in range(T_tab)]
    tab = season.build_table(names, groups=groups, points=(3, 1))
    tab["start_points"] = rng.integers(0, 30, T_tab).astype(np.int32)
    tab["start_goals_for"] = rng.integers(0, 40, T_tab).astype(np.int32)
    tab["start_goals_against"] = rng.integers(0, 40, T_tab).astype(np.int32)
    h = rng.integers(0, T_tab, F)
    a = (h + rng.integers(1, T_tab, F)) % T_tab
    hs, as_ = season.fixture_slots(tab, [names[i] for i in h], [names[i] for i in a])
    fx = {"home_team": team_of_slot[hs].astype(np.uint16), "away_team": team_of_slot[as_].astype(np.uint16)}
    if model in ("neutral", "neutral_wc"):
        fx["neutral_venue"] = (rng.random(F) < 0.4).astype(np.uint8)
    if model == "neutral_wc":
        fx["home_conf"] = rng.integers(0, Cf, F).astype(np.uint8)
        fx["away_conf"] = rng.integers(0, Cf, F).astype(np.uint8)
    return s, fx, hs, as_, tab


def _run(model, s, fx, hs, as_, tab, G, R, seed, first_draw=0, raw=True):
    from bpl_next_b200 import simulate_table

    out = simulate_table(model, _dev(s), _dev(dict(fx, home_slot=hs, away_slot=as_)), _dev_table(tab), G, R, seed,
                         first_draw=first_draw, want_positions=raw, want_scores=raw)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


REPLAY = [(1, 15, 2, False, 5), (7, 4, 20, False, 60), (7, 15, 20, True, 60), (1, 15, 64, True, 100),
          (7, 15, 64, False, 100)]


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("R,G,T_tab,grouped,F", REPLAY)
def test_exact_replay(model, R, G, T_tab, grouped, F):
    """Every kernel score equals the oracle's on the same Philox words, except (simulation, fixture) pairs whose oracle
    margin is below 1e-5 (float32 rounding at a cumulative boundary), at most 0.1 % of them; the histograms and the raw
    positions equal, integer for integer, the oracle's ranking of the kernel's own scores.  S = 149 draws: N is ragged."""
    S, seed = 149, 1000 + R * 100 + T_tab
    s, fx, hs, as_, tab = _case(model, S, T_tab, grouped, F, seed)
    k = _run(model, s, fx, hs, as_, tab, G, R, seed)
    o = osim.simulate(model, s, fx, hs, as_, tab, G, R, seed)
    assert k["invalid"][0] == 0 and o["invalid"] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    diff = (kh != o["home"]) | (ka != o["away"])
    small = o["margin"] < 1e-5
    assert not (diff & ~small).any(), np.argwhere(diff & ~small)[:5]
    assert diff.sum() <= 1e-3 * diff.size
    r = osim.rank_scores(tab, hs, as_, kh, ka, o["keys"])
    np.testing.assert_array_equal(k["positions"], r["positions"])
    np.testing.assert_array_equal(k["position_counts"], r["position_counts"])
    np.testing.assert_array_equal(k["points_counts"], r["points_counts"])
    assert k["position_counts"].sum() == S * R * T_tab


def test_draw_ranges_and_seeds():
    """Draws [0, 17) and [17, 50) with first_draw: counts sum to the single call's bit for bit and the raw rows
    concatenate to its rows; the same seed repeats, another seed differs."""
    s, fx, hs, as_, tab = _case("neutral_wc", 50, 12, True, 40, seed=5)
    full = _run("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=99)
    parts = [_run("neutral_wc", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, 15, 3, seed=99, first_draw=lo)
             for lo, hi in ((0, 17), (17, 50))]
    for key in ("position_counts", "points_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key])
    for key in ("positions", "scores"):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]))
    again = _run("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=99)
    for key in ("position_counts", "points_counts", "positions", "scores"):
        np.testing.assert_array_equal(full[key], again[key])
    other = _run("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=100)
    assert not np.array_equal(full["scores"], other["scores"])
    # the counts do not depend on whether the raw outputs are written
    noraw = _run("neutral_wc", s, fx, hs, as_, tab, 15, 3, seed=99, raw=False)
    np.testing.assert_array_equal(full["position_counts"], noraw["position_counts"])


def test_cells_against_the_predict_path():
    """One neutral-venue WC fixture, N = 2^22 simulations: every cell's frequency within 5 sigma of the score grid of
    the same draws (bplx_score_grid, the average of the per-draw grids)."""
    from bpl_next_b200 import score_grid

    s, fx, hs, as_, tab = _case("neutral_wc", 64, 2, False, 1, seed=21)
    fx["neutral_venue"][:] = 1
    N = 64 * 65536
    k = _run("neutral_wc", s, fx, hs, as_, tab, 15, 65536, seed=3)
    grid, _ = score_grid("neutral_wc", _dev(s), _dev(fx), 15)
    p = grid[0].double().cpu().numpy()
    counts = np.bincount(k["scores"][:, 0, 0].astype(np.int64) * 16 + k["scores"][:, 0, 1], minlength=256)
    counts = counts.reshape(16, 16)
    sig = np.sqrt(N * p * (1 - p))
    assert (np.abs(counts - N * p) <= 5 * sig + 1).all(), np.abs(counts - N * p).max()


def test_expected_points_against_the_outcome_probabilities():
    """A four-team round robin at N = 2^20: expected final points = start + sum over the team's fixtures of
    3 p_win + 1 p_draw from bplx_score_grid's outcome probabilities of the same draws, within 5 Monte-Carlo SE."""
    from bpl_next_b200 import score_grid

    s, _, _, _, _ = _case("dixon_coles", 64, 4, False, 6, seed=31)
    names = ["S0", "S1", "S2", "S3"]
    tab = season.build_table(names, {"home_team": ["S0"], "away_team": ["S1"], "home_goals": [1], "away_goals": [1]})
    pairs = [(i, j) for i in range(4) for j in range(4) if i < j]
    hs, as_ = season.fixture_slots(tab, [names[i] for i, _ in pairs], [names[j] for _, j in pairs])
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16)}
    R = 16384
    N = 64 * R
    k = _run("dixon_coles", s, fx, hs, as_, tab, 15, R, seed=8, raw=False)
    pr = season.probabilities(tab, k["position_counts"], k["points_counts"], N)
    _, out = score_grid("dixon_coles", _dev(s), _dev(fx), 15)
    out = out.double().cpu().numpy()
    want = tab["start_points"].astype(np.float64)
    for f, (i, j) in enumerate(pairs):
        want[i] += 3 * out[f, 0] + out[f, 1]
        want[j] += 3 * out[f, 2] + out[f, 1]
    b = np.arange(pr["points_proba"].shape[1])
    var = pr["points_proba"] @ b ** 2 - (pr["points_proba"] @ b) ** 2
    se = np.sqrt(var / N)
    assert (np.abs(pr["expected_points"] - want) <= 5 * se).all(), (pr["expected_points"] - want) / se


def _raw_call(model, s, fx, hs, as_, tab, G, R):
    """bplx_simulate_table called directly (no Python-side checks) on one table without groups; returns (status,
    invalid count)."""
    from bpl_next_b200 import problem

    lib = _abi.lib()
    keep = []
    ptr = problem._device_ptr_fn(keep)
    st = problem._samples_struct(model, _dev(s), ptr)
    ft = problem._fixtures_struct(_dev(fx), ptr)
    t = problem._table_struct(dict(_dev_table(tab), group=None), ptr)
    slots = _dev({"h": hs, "a": as_})
    pc = torch.empty((t.num_slots, t.num_positions), dtype=torch.int64, device="cuda")
    bc = torch.empty((t.num_slots, t.num_points_bins), dtype=torch.int64, device="cuda")
    inv = torch.empty(1, dtype=torch.int64, device="cuda")
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    rc = lib.bplx_simulate_table(C.byref(st), C.byref(ft), ptr(slots["h"]), ptr(slots["a"]), C.byref(t), G, R, 1, 0,
                                 ptr(pc), ptr(bc), None, None, ptr(inv), ptr(ws), ws.numel(), None)
    torch.cuda.synchronize()
    return rc, int(inv.item())


def test_tau_clamp_invalid_draws_and_refusals():
    from bpl_next_b200 import DixonColesMatchPredictor, simulate_table

    # corr_coef = 5: tau(1, 1) = 1 - 5 < 0 and tau(0, 0) = 1 - 5 lh la < 0 for these rates: never drawn
    s, fx, hs, as_, tab = _case("dixon_coles", 16, 3, False, 6, seed=41)
    s["corr_coef"][:] = 5.0
    k = _run("dixon_coles", s, fx, hs, as_, tab, 15, 500, seed=2)
    sc = k["scores"].astype(np.int64)
    lh, la = op.expected_goals("dixon_coles", s, fx["home_team"], fx["away_team"])
    t00_zero = np.repeat(1.0 - 5.0 * lh * la <= 0.0, 500, axis=0)  # [N, F]
    assert t00_zero.mean() > 0.9
    assert not ((sc[..., 0] == 1) & (sc[..., 1] == 1)).any()
    assert not ((sc[..., 0] == 0) & (sc[..., 1] == 0) & t00_zero).any()
    assert k["invalid"][0] == 0

    # non-finite rates: the simulations of those draws are invalid, left out of the counts, their rows 0xFF
    s, fx, hs, as_, tab = _case("dixon_coles", 12, 6, False, 15, seed=42)
    s["attack"][3, fx["home_team"][0]] = np.inf
    s["defence"][7, fx["away_team"][2]] = np.nan
    o = osim.simulate("dixon_coles", s, fx, hs, as_, tab, 15, 5, seed=4)
    k = _run("dixon_coles", s, fx, hs, as_, tab, 15, 5, seed=4)
    assert k["invalid"][0] == o["invalid"] == 10
    np.testing.assert_array_equal((k["positions"] == 255).all(axis=1), ~o["valid"])
    assert k["position_counts"].sum() == (12 * 5 - 10) * 6

    # ... and the predictor raises
    m = DixonColesMatchPredictor()
    m.teams = np.array([f"S{i}" for i in range(9)])
    m._teams_dict = {t: i for i, t in enumerate(m.teams)}
    m.attack, m.defence, m.home_advantage, m.corr_coef = s["attack"], s["defence"], s["home_advantage"], s["corr_coef"]
    bad1, bad2 = m.teams[fx["home_team"][0]], m.teams[fx["away_team"][2]]
    other = next(t for t in m.teams if t not in (bad1, bad2))
    with pytest.raises(ValueError, match="non-finite"):
        m.simulate_table({"home_team": [bad1, bad2], "away_team": [other, other]}, num_sims_per_draw=2, random_state=1)

    # refusals: DYNAMIC, more than 64 slots, max_goals outside [1, 63], sims_per_draw < 1, a slot outside the table
    s, fx, hs, as_, tab = _case("dixon_coles", 8, 4, False, 6, seed=43)
    with pytest.raises(_abi.BplxError):
        _run("dynamic", s, fx, hs, as_, tab, 15, 2, seed=1)
    for G, R in ((0, 2), (64, 2), (15, 0)):
        with pytest.raises(_abi.BplxError):
            _run("dixon_coles", s, fx, hs, as_, tab, G, R, seed=1)
    big = dict(tab, start_points=np.zeros(65, np.int32), start_goals_for=np.zeros(65, np.int32),
               start_goals_against=np.zeros(65, np.int32))
    with pytest.raises(ValueError, match="at most 64"):
        _run("dixon_coles", s, fx, hs, as_, big, 15, 2, seed=1)
    assert _raw_call("dixon_coles", s, fx, hs, as_, big, 15, 2)[0] == _abi.E_UNSUPPORTED
    bad = as_.copy()
    bad[1] = 4
    with pytest.raises(ValueError, match="slot 4"):
        _run("dixon_coles", s, fx, hs, bad, tab, 15, 2, seed=1)
    rc, inv = _raw_call("dixon_coles", s, fx, hs, bad, tab, 15, 2)  # the kernel never reads or writes past the table
    assert rc == _abi.OK and inv == 8 * 2


def _take(td, ix):
    return {k: ([v[i] for i in ix] if isinstance(v, list) else np.asarray(v)[ix]) for k, v in td.items()}


@pytest.fixture(scope="module")
def dc_half_season():
    from bpl_next_b200 import DixonColesMatchPredictor

    td = datasets.dummy_data()
    first, rest = _take(td, np.arange(190)), _take(td, np.arange(190, 380))
    m = DixonColesMatchPredictor().fit(first, num_warmup=300, num_samples=500, mcmc_kwargs={"num_chains": 8})
    return m, first, rest


def test_end_to_end_league(dc_half_season, monkeypatch):
    """DixonColes fit of the first 190 matches of dummy_data (8 chains), the other 190 simulated from the table of the
    first 190: probabilities sum to 1, expected points = start + sum (3 p_win + p_draw) of predict_outcome_proba within
    5 Monte-Carlo SE, a fixed random_state repeats exactly, and ranges of draws do not change the results."""
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor, predictors

    m, first, rest = dc_half_season
    fx = {"home_team": rest["home_team"], "away_team": rest["away_team"]}
    res = m.simulate_table(fx, played=first, num_sims_per_draw=4, random_state=5)
    S = m.attack.shape[0]
    N = S * 4
    assert res["num_simulations"] == N and res["sims_per_draw"] == 4 and res["seed"] == 5
    assert res["teams"] == sorted(set(first["home_team"]) | set(first["away_team"]))
    pp, bp = res["position_proba"], res["points_proba"]
    assert pp.shape == (20, 20)
    np.testing.assert_allclose(pp.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(pp.sum(axis=0), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(bp.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    start = season.build_table(res["teams"], first)["start_points"]
    np.testing.assert_array_equal(res["start_points"], start)
    out = m.predict_outcome_proba(rest["home_team"], rest["away_team"])
    slot = {t: i for i, t in enumerate(res["teams"])}
    want = start.astype(np.float64)
    for f, (h, a) in enumerate(zip(rest["home_team"], rest["away_team"])):
        want[slot[h]] += 3 * out["home_win"][f] + out["draw"][f]
        want[slot[a]] += 3 * out["away_win"][f] + out["draw"][f]
    b = np.arange(bp.shape[1])
    se = np.sqrt((bp @ b ** 2 - (bp @ b) ** 2) / N)
    assert (np.abs(res["expected_points"] - want) <= 5 * se).all()

    again = m.simulate_table(fx, played=first, num_sims_per_draw=4, random_state=5)
    for key in ("position_proba", "points_proba", "expected_points"):
        np.testing.assert_array_equal(res[key], again[key])
    monkeypatch.setattr(predictors, "SIM_OUTPUT_BYTES", 4 * (20 + 2 * 190) * 333)  # ranges of 333 draws
    raw = m.simulate_table(fx, played=first, num_sims_per_draw=4, random_state=5, return_simulations=True)
    for key in ("position_proba", "points_proba", "expected_points"):
        np.testing.assert_array_equal(res[key], raw[key])
    assert raw["positions"].shape == (N, 20) and raw["positions"].dtype == np.uint8
    assert raw["home_score"].shape == (190, N) and raw["away_score"].shape == (190, N)
    counts = np.stack([np.bincount(raw["positions"][:, t], minlength=20) for t in range(20)])
    np.testing.assert_array_equal(counts, np.rint(pp * N).astype(np.int64))

    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().simulate_table(fx)


def test_group_stage_neutral_wc():
    """A NeutralWC fit; two groups of four at neutral venues with confederations: positions are per group (P = 4), each
    group's positions are filled exactly once per simulation."""
    from bpl_next_b200 import NeutralDixonColesMatchPredictorWC

    m = NeutralDixonColesMatchPredictorWC().fit(datasets.neutral_dummy_data(), num_warmup=150, num_samples=100,
                                               mcmc_kwargs={"num_chains": 8})
    teams = [str(i) for i in range(8)]
    groups = {t: "A" if int(t) < 4 else "B" for t in teams}
    pairs = [(a, b) for g in ("A", "B") for a in teams for b in teams if groups[a] == groups[b] == g and int(a) < int(b)]
    fx = {"home_team": [a for a, _ in pairs], "away_team": [b for _, b in pairs],
          "home_conf": [str(int(a) // 4) for a, _ in pairs], "away_conf": [str(int(b) // 4) for _, b in pairs],
          "neutral_venue": [1] * len(pairs)}
    res = m.simulate_table(fx, groups=groups, num_sims_per_draw=8, random_state=3)
    pp = res["position_proba"]
    assert res["teams"] == teams and res["groups"] == ["A"] * 4 + ["B"] * 4 and pp.shape == (8, 4)
    np.testing.assert_allclose(pp.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(pp[:4].sum(axis=0), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(pp[4:].sum(axis=0), 1.0, rtol=0, atol=1e-12)
    assert res["points_proba"].shape == (8, 3 * 3 + 1)
