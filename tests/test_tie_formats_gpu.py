"""Knockout tie formats on the GPU: a bracket of format-0 ties through bplx_simulate_tournament_ex is bit-identical to
bplx_simulate_tournament; the kernel replayed exactly by the float64 oracle with formats mixed; draw ranges and seeds;
a two-legged and an extra-time tie at N = 2^22 against the per-draw closed form and the reversed fixture's grid; a
league with play-offs and the Champions League shape through the predictors; refusals."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

from bpl_next_b200 import _abi, problem, season
from oracle import tournament
from tests.test_score_grid_gpu import make_samples
from tests.test_simulate_gpu import _dev, _dev_table
from tests.test_tournament_gpu import REPLAY, _case, _raw_call, _run, _wc_predictor, _world_cup_48

pytestmark = pytest.mark.gpu

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _timing_script():
    spec = importlib.util.spec_from_file_location("tournament_time",
                                                  os.path.join(_ROOT, "scripts", "tournament_time.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _mixed_formats(br):
    """Every third tie one match, the others two legs, or one match with extra time where the venue is neutral."""
    nv = np.asarray(br["neutral_venue"])
    fmt = [0 if k % 3 == 2 else (1 if nv[k] else 2) for k in range(len(br["round"]))]
    return dict(br, tie_format=np.asarray(fmt, np.uint8))


def _legacy(model, s, fx, hs, as_, tab, br, G, R, seed):
    """bplx_simulate_tournament with every output, on the arguments problem.simulate_tournament passes."""
    lib = _abi.lib()
    keep = []
    ptr = problem._device_ptr_fn(keep)
    st = problem._samples_struct(model, _dev(s), ptr)
    dfx = _dev(dict(fx, home_slot=hs, away_slot=as_))
    ft = problem._fixtures_struct(dfx, ptr)
    t = problem._table_struct(_dev_table(tab), ptr)
    b = problem._bracket_struct(br, keep)
    T, K, N = t.num_slots, b.num_ties, s["attack"].shape[0] * R
    ws = torch.empty(int(lib.bplx_simulate_tournament_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t),
                                                                     C.byref(b))), dtype=torch.uint8, device="cuda")
    i64, u8 = dict(dtype=torch.int64, device="cuda"), dict(dtype=torch.uint8, device="cuda")
    out = {"position_counts": torch.empty((T, t.num_positions), **i64),
           "points_counts": torch.empty((T, t.num_points_bins), **i64),
           "reach_counts": torch.empty((T, b.num_rounds), **i64), "win_counts": torch.empty((T, b.num_rounds), **i64),
           "positions": torch.empty((N, T), **u8), "scores": torch.empty((N, len(hs), 2), **u8),
           "ko_entrants": torch.empty((N, K, 2), **u8), "ko_scores": torch.empty((N, K, 2), **u8),
           "ko_winners": torch.empty((N, K), **u8), "invalid": torch.empty(1, **i64)}
    _abi.check(lib.bplx_simulate_tournament(C.byref(st), C.byref(ft), ptr(dfx["home_slot"]), ptr(dfx["away_slot"]),
                                            C.byref(t), C.byref(b), G, R, seed, 0,
                                            *(ptr(v) for v in out.values()), ptr(ws), ws.numel(), None))
    return {k: v.cpu().numpy() for k, v in out.items()}


def test_format_0_is_bitwise_the_legacy_call():
    """The 48-team World Cup, every tie format 0, through _ex (problem.simulate_tournament) and through
    bplx_simulate_tournament with the same seed: every output the same bits; nothing goes to extra time."""
    S, R = 96, 3
    teams, groups, fx, ties, best = _world_cup_48()
    s = make_samples("neutral_wc", S, 60, 6, seed=81)
    tab = season.build_table(teams, groups=groups)
    hs, as_ = season.fixture_slots(tab, fx["home_team"], fx["away_team"])
    idx = {t: i for i, t in enumerate(teams)}
    fxa = {"home_team": np.asarray([idx[t] for t in fx["home_team"]], np.uint16),
           "away_team": np.asarray([idx[t] for t in fx["away_team"]], np.uint16),
           "home_conf": np.asarray([int(c[1:]) for c in fx["home_conf"]], np.uint8),
           "away_conf": np.asarray([int(c[1:]) for c in fx["away_conf"]], np.uint8),
           "neutral_venue": np.asarray(fx["neutral_venue"], np.uint8)}
    br = season.build_bracket(tab, ties, best)
    br["slot_team"] = np.arange(48, dtype=np.uint16)
    br["slot_conf"] = (np.arange(48) % 6).astype(np.uint8)
    assert (br["tie_format"] == 0).all()
    new = _run("neutral_wc", s, fxa, hs, as_, tab, br, 15, R, seed=23)
    old = _legacy("neutral_wc", s, fxa, hs, as_, tab, br, 15, R, seed=23)
    assert old["invalid"][0] == 0
    for k, v in old.items():
        np.testing.assert_array_equal(new[k], v, err_msg=k)
    assert (new["ko_extra"] == tournament.NOT_PLAYED).all()
    d = new["decided_counts"]
    assert (d[:, 1] == 0).all() and (d.sum(axis=1) == S * R).all() and d[:, 2].sum() > 0


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("R,T_tab,grouped,best,F", REPLAY)
def test_exact_replay_with_formats(model, R, T_tab, grouped, best, F):
    """Formats 0, 1 and 2 mixed: kernel scores of every match, ko_extra and winners equal the oracle's on the same
    Philox words except where one of the oracle's margins is below 1e-5 (test_exact_replay's bound); entrants and every
    count equal, integer for integer, resolve_bracket applied to the kernel's own raw rows.  S = 149: N is ragged."""
    S, seed = 149, 3000 + R * 100 + T_tab + F
    s, fx, hs, as_, tab, br = _case(model, S, T_tab, grouped, F, seed, best=best)
    br = _mixed_formats(br)
    k = _run(model, s, fx, hs, as_, tab, br, 15, R, seed)
    o = tournament.simulate_tournament(model, s, fx if F else None, hs, as_, tab, br, 15, R, seed)
    assert k["invalid"][0] == 0 and o["invalid"] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    gdiff = (kh != o["home"]) | (ka != o["away"])
    assert not (gdiff & ~(o["margin"] < 1e-5)).any(), np.argwhere(gdiff & ~(o["margin"] < 1e-5))[:5]
    kk = {x: k[x].astype(np.int64) for x in ("ko_scores", "ko_winners", "ko_entrants", "ko_extra")}
    same_ent = (kk["ko_entrants"] == o["ko_entrants"]).all(axis=2)
    diff = ((kk["ko_scores"] != o["ko_scores"]).any(axis=2) | (kk["ko_winners"] != o["ko_winners"])
            | (kk["ko_extra"] != o["ko_extra"]).any(axis=2))
    small_ko = ((o["ko_margin"] < 1e-5) | (o["leg2_margin"] < 1e-5) | (o["extra_time_margin"] < 1e-5)
                | (o["decider_margin"] < 1e-5))
    assert not (diff & same_ent & ~small_ko).any(), np.argwhere(diff & same_ent & ~small_ko)[:5]
    assert gdiff.sum() <= max(1, 1e-3 * gdiff.size) and (diff | ~same_ent).sum() <= max(2, 1e-3 * diff.size)
    ent = kk["ko_entrants"]
    through = kk["ko_winners"] == ent[:, :, 0]
    r = tournament.resolve_bracket(tab, hs, as_, br, kh, ka, o["keys"], kk["ko_scores"][:, :, 0],
                                   kk["ko_scores"][:, :, 1], through, ko_extra=kk["ko_extra"])
    for key in ("ko_entrants", "ko_winners", "ko_extra", "reach_counts", "win_counts", "decided_counts", "positions",
                "position_counts", "points_counts"):
        np.testing.assert_array_equal(k[key], r[key], err_msg=key)
    K, N = len(br["round"]), S * R
    assert k["reach_counts"].sum() == 2 * K * N and k["win_counts"].sum() == K * N
    assert (k["decided_counts"].sum(axis=1) == N).all()
    fmt = br["tie_format"]
    assert (k["decided_counts"][fmt == 0, 1] == 0).all()
    assert (k["ko_extra"][:, fmt != 2, :2] == tournament.NOT_PLAYED).all()
    assert (k["ko_extra"][:, fmt == 0] == tournament.NOT_PLAYED).all()
    played = k["ko_extra"][:, :, 2] != tournament.NOT_PLAYED
    np.testing.assert_array_equal(played.sum(axis=0), k["decided_counts"][:, 1:].sum(axis=1) * (fmt != 0))


def test_draw_ranges_and_seeds_with_formats():
    s, fx, hs, as_, tab, br = _case("neutral_wc", 50, 16, True, 40, seed=5, best=True)
    br = _mixed_formats(br)
    full = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=99)
    parts = [_run("neutral_wc", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, br, 15, 3, seed=99,
                  first_draw=lo) for lo, hi in ((0, 17), (17, 50))]
    for key in ("position_counts", "points_counts", "reach_counts", "win_counts", "decided_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key], err_msg=key)
    for key in ("positions", "scores", "ko_entrants", "ko_scores", "ko_winners", "ko_extra"):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]), err_msg=key)
    other = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=100)
    assert not np.array_equal(full["ko_extra"], other["ko_extra"])
    noraw = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=99, raw=False)
    for key in ("reach_counts", "win_counts", "decided_counts"):
        np.testing.assert_array_equal(full[key], noraw[key])


@pytest.mark.parametrize("model,fmt,neutral", [("dixon_coles", "two_legs", 0), ("neutral_wc", "extra_time", 1)])
def test_one_tie_against_the_closed_form(model, fmt, neutral):
    """One tie, N = 2^22: P(A through), P(extra time) and P(penalties) within 5 sigma of the mean over draws of the
    float64 closed form; for two legs, every cell of the leg-2 score (B at home) within 5 sigma of score_grid of the
    reversed fixture."""
    from bpl_next_b200 import score_grid

    S, R, G = 64, 65536, 15
    N = S * R
    s = make_samples(model, S, 5, 4, seed=27)
    tab = season.build_table(["S0", "S1"])
    tab["num_points_bins"], tab["num_positions"] = 1, 2
    br = season.build_bracket(tab, [{"id": "t", "round": "F", "home": ("team", "S0"), "away": ("team", "S1"),
                                     "neutral_venue": neutral, "format": fmt}])
    br["slot_team"] = np.array([3, 1], np.uint16)
    br["slot_conf"] = np.array([2, 0], np.uint8)
    e = np.zeros(0, np.uint8)
    k = _run(model, s, {}, e, e, tab, br, G, R, seed=8)
    assert k["invalid"][0] == 0
    code = season.TIE_FORMATS[fmt]
    p_through, p_et, p_pen = (x.mean() for x in tournament.tie_closed_form(model, s, 3, 1, code, G, neutral, 2, 0))
    d = k["decided_counts"][0]
    for share, p in (((k["ko_winners"][:, 0] == 0).mean(), p_through), (d[1:].sum() / N, p_et), (d[2] / N, p_pen)):
        assert abs(share - p) <= 5 * np.sqrt(p * (1 - p) / N), (share, p)
    if code == tournament.TWO_LEGS:
        fx = {"home_team": np.array([1], np.uint16), "away_team": np.array([3], np.uint16)}
        grid, _ = score_grid(model, _dev(s), _dev(fx), G)
        pc = grid[0].double().cpu().numpy()
        b_goals, a_goals = k["ko_extra"][:, 0, 1].astype(np.int64), k["ko_extra"][:, 0, 0].astype(np.int64)
        counts = np.bincount(b_goals * 16 + a_goals, minlength=256).reshape(16, 16)
        assert (np.abs(counts - N * pc) <= 5 * np.sqrt(N * pc * (1 - pc)) + 1).all()
    else:
        assert (k["ko_extra"][:, 0, :2] == tournament.NOT_PLAYED).all()


def _dc_predictor(T, S=256, seed=91):
    from bpl_next_b200 import DixonColesMatchPredictor

    s = make_samples("dixon_coles", S, T, 1, seed=seed)
    m = DixonColesMatchPredictor()
    m.teams = [f"T{i:02d}" for i in range(T)]
    m._teams_dict = {t: i for i, t in enumerate(m.teams)}
    m.attack, m.defence, m.home_advantage, m.corr_coef = s["attack"], s["defence"], s["home_advantage"], s["corr_coef"]
    return m


def _check_bracket_result(res, ties):
    N = res["num_simulations"]
    np.testing.assert_allclose(res["champion_proba"].sum(), 1.0, rtol=0, atol=1e-12)
    rounds = [t["round"] for t in ties]
    for r, label in enumerate(res["rounds"]):
        np.testing.assert_allclose(res["reach_proba"][:, r].sum(), 2.0 * rounds.count(label), rtol=0, atol=1e-9)
    np.testing.assert_allclose(res["decided_proba"].sum(axis=1), 1.0, rtol=0, atol=1e-12)
    assert res["tie_ids"] == [t["id"] for t in ties]
    return N


def test_league_with_play_offs_end_to_end():
    """24 teams, 48 remaining fixtures; play-offs 6th v 3rd and 5th v 4th over two legs (the lower-placed team at home
    first), then a final with extra time: only teams placed 3rd-6th ever reach it."""
    m = _dc_predictor(24)
    teams = m.teams
    rng = np.random.default_rng(3)
    h = rng.integers(0, 24, 48)
    a = (h + rng.integers(1, 24, 48)) % 24
    fx = {"home_team": [teams[i] for i in h], "away_team": [teams[i] for i in a]}
    played = {"home_team": teams[:12], "away_team": teams[12:], "home_goals": rng.integers(0, 4, 12),
              "away_goals": rng.integers(0, 4, 12)}
    ties = [{"id": "p1", "round": "semi", "home": ("group", None, 5), "away": ("group", None, 2), "format": "two_legs"},
            {"id": "p2", "round": "semi", "home": ("group", None, 4), "away": ("group", None, 3), "format": "two_legs"},
            {"id": "f", "round": "final", "home": ("winner", "p1"), "away": ("winner", "p2"), "format": "extra_time"}]
    res = m.simulate_tournament(fx, ties, played=played, teams=teams, num_sims_per_draw=16, random_state=5,
                                return_simulations=True)
    N = _check_bracket_result(res, ties)
    assert res["ko_extra"].shape == (N, 3, 4)
    pos = res["positions"]
    final = res["ko_entrants"][:, 2].astype(np.int64)
    placed = np.take_along_axis(pos, final, axis=1)
    assert ((placed >= 2) & (placed <= 5)).all()
    np.testing.assert_array_equal(np.take_along_axis(pos, res["ko_entrants"][:, 0].astype(np.int64), axis=1),
                                  np.broadcast_to([5, 2], (N, 2)))
    d = res["decided_proba"]
    assert d[0, 1] > 0 and d[0, 2] > 0 and d[2, 1] > 0


def test_champions_league_end_to_end():
    """The timing script's Champions League shape on a NeutralWC predictor: 36-team league phase, play-offs 9-24,
    two-legged ties through the semi-finals, a neutral final with extra time."""
    tt = _timing_script()
    m = _wc_predictor()
    teams = m.teams[:36]
    conf = {t: f"C{i % 6}" for i, t in enumerate(teams)}
    hs = np.repeat(np.arange(36), 4)
    as_ = (hs + np.tile(np.arange(1, 5), 36)) % 36
    fx = {"home_team": [teams[i] for i in hs], "away_team": [teams[i] for i in as_],
          "home_conf": [conf[teams[i]] for i in hs], "away_conf": [conf[teams[i]] for i in as_],
          "neutral_venue": [0] * len(hs)}
    ties = tt.champions_league_ties()
    assert len(ties) == 23 and len(fx["home_team"]) == 144
    res = m.simulate_tournament(fx, ties, teams=teams, num_sims_per_draw=8, random_state=2)
    _check_bracket_result(res, ties)
    assert res["rounds"] == ["PO", "R16", "QF", "SF", "F"]
    # positions 25-36 go out in the league phase; the top 8 skip the play-offs
    top8 = res["position_proba"][:, :8].sum(axis=1)
    out = res["position_proba"][:, 24:].sum(axis=1)
    np.testing.assert_allclose(res["reach_proba"][:, 0], 1.0 - top8 - out, rtol=0, atol=1e-9)
    d = res["decided_proba"]
    assert (d[:22, 0] > 0.5).all() and (d[:22, 1] > 0).all() and d[22, 1] > 0


def test_refusals():
    s, fx, hs, as_, tab, br = _case("dixon_coles", 8, 8, False, 0, seed=71)
    bad = dict(br, tie_format=np.full(len(br["round"]), 3, np.uint8))
    with pytest.raises(_abi.BplxError, match="format 3"):
        _run("dixon_coles", s, fx, hs, as_, tab, bad, 15, 2, seed=1)
    nv = dict(br, tie_format=np.full(len(br["round"]), 2, np.uint8), neutral_venue=np.zeros_like(br["neutral_venue"]))
    nv["neutral_venue"][1] = 1
    with pytest.raises(_abi.BplxError, match="neutral venue"):
        _run("dixon_coles", s, fx, hs, as_, tab, nv, 15, 2, seed=1)
    nv["neutral_venue"][1] = 0
    out = _run("dixon_coles", s, fx, hs, as_, tab, nv, 15, 2, seed=1)
    assert out["invalid"][0] == 0 and (out["decided_counts"].sum(axis=1) == 16).all()
    assert _raw_call("dixon_coles", s, tab, br) == _abi.OK  # the legacy entry point, unchanged
    # through Python: build_bracket and the predictor refuse before any call
    m = _dc_predictor(8)
    ties = [{"id": "f", "round": "F", "home": ("team", "T00"), "away": ("team", "T01"), "neutral_venue": 1,
             "format": "two_legs"}]
    with pytest.raises(ValueError, match="neutral venue"):
        m.simulate_tournament(None, ties)
    ties[0].update(neutral_venue=0, format="replay")
    with pytest.raises(ValueError, match="unknown format"):
        m.simulate_tournament(None, ties)
