"""Tournament simulation on the GPU: the kernel replayed exactly by the float64 oracle (oracle/tournament.py) on the
same Philox words, the group stage bit-identical to bplx_simulate_table, draw ranges and seeds, the decider and the tie
scores against the per-draw grids, a knockout-only bracket, the 48-team World Cup format through the predictor, and
refusals."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from bpl_next_b200 import _abi, season
from oracle import predict as op
from oracle import tournament
from tests.test_score_grid_gpu import make_samples
from tests.test_simulate_gpu import _dev, _dev_table

pytestmark = pytest.mark.gpu


def _alloc(labels, count):
    out = {}
    for sub in itertools.combinations(labels, count):
        r = len(out) % count
        out[frozenset(sub)] = list(sub[r:] + sub[:r])
    return out


def _knockout(entrants, third_place=True, neutral=None):
    """Ties pairing ``entrants`` in order, then the winners round by round; a third-place match before the final."""
    ties, prev, r = [], list(entrants), 0
    while len(prev) > 1:
        cur = []
        for k in range(0, len(prev), 2):
            tid = f"t{len(ties)}"
            ties.append({"id": tid, "round": f"r{r}", "home": prev[k], "away": prev[k + 1],
                         "neutral_venue": int(neutral[len(ties) % len(neutral)]) if neutral is not None else 0})
            cur.append(("winner", tid))
        if len(cur) == 1 and third_place and len(ties) >= 3:
            final = ties.pop()
            a, b = final["home"][1], final["away"][1]
            ties.append({"id": "third", "round": "third", "home": ("loser", a), "away": ("loser", b)})
            ties.append(final)
        prev, r = cur, r + 1
    return ties


def _case(model, S, T_tab, grouped, F, seed, Cf=4, best=False):
    """Samples for T_tab + 3 model teams, T_tab slots mapped to a random subset of them, a random start, F random
    fixtures between slots; an eight-entrant bracket with a third-place match: group winners, runners-up and (with
    ``best``) the two best thirds through an allocation table, or the top eight of a single table."""
    T = T_tab + 3
    s = make_samples(model, S, T, Cf, seed=seed)
    rng = np.random.default_rng(seed + 1)
    team_of_slot = rng.permutation(T)[:T_tab]
    names = [f"S{i}" for i in range(T_tab)]
    groups = [f"g{i // 4}" for i in range(T_tab)] if grouped else None
    tab = season.build_table(names, groups=groups, points=(3, 1))
    tab["start_points"] = rng.integers(0, 5, T_tab).astype(np.int32)
    tab["start_goals_for"] = rng.integers(0, 6, T_tab).astype(np.int32)
    tab["start_goals_against"] = rng.integers(0, 6, T_tab).astype(np.int32)
    fx, hs, as_ = {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8)
    if F:
        h = rng.integers(0, T_tab, F)
        a = (h + rng.integers(1, T_tab, F)) % T_tab
        hs, as_ = season.fixture_slots(tab, [names[i] for i in h], [names[i] for i in a])
        fx = {"home_team": team_of_slot[hs].astype(np.uint16), "away_team": team_of_slot[as_].astype(np.uint16)}
        if model in ("neutral", "neutral_wc"):
            fx["neutral_venue"] = (rng.random(F) < 0.4).astype(np.uint8)
        if model == "neutral_wc":
            fx["home_conf"] = rng.integers(0, Cf, F).astype(np.uint8)
            fx["away_conf"] = rng.integers(0, Cf, F).astype(np.uint8)
    else:
        season._size_histograms(tab)
    bspec = None
    if grouped:
        L = tab["group_labels"]
        ent = [("group", g, 0) for g in L] + [("group", g, 1) for g in L[:2]]
        if best:
            ent += [("best", 0), ("best", 1)]
            bspec = {"position": 2, "count": 2, "allocation": _alloc(L, 2)}
        else:
            ent += [("group", g, 1) for g in L[2:4]]
        ent = ent[:8]
    else:
        ent = [("group", None, p) for p in range(8)] if F else [("team", n) for n in names[:8]]
    ties = _knockout(ent, neutral=[0, 1, 1])
    br = season.build_bracket(tab, ties, bspec)
    br["slot_team"] = team_of_slot.astype(np.uint16)
    if model == "neutral_wc":
        br["slot_conf"] = rng.integers(0, Cf, T_tab).astype(np.uint8)
    return s, fx, hs, as_, tab, br


def _run(model, s, fx, hs, as_, tab, br, G, R, seed, first_draw=0, raw=True):
    from bpl_next_b200 import simulate_tournament

    dfx = _dev(dict(fx, home_slot=hs, away_slot=as_)) if len(hs) else {}
    out = simulate_tournament(model, _dev(s), dfx, _dev_table(tab), br, G, R, seed, first_draw=first_draw,
                              want_positions=raw, want_scores=raw, want_knockout=raw)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


REPLAY = [(1, 15, True, True, 40), (7, 15, True, False, 40), (7, 12, False, False, 30), (1, 8, False, False, 0)]


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral", "neutral_wc"])
@pytest.mark.parametrize("R,T_tab,grouped,best,F", REPLAY)
def test_exact_replay(model, R, T_tab, grouped, best, F):
    """Kernel scores and winners equal the oracle's on the same Philox words except where the oracle's score or
    decider margin is below 1e-5 (at most 0.1 % of pairs); entrants and every count equal, integer for integer,
    resolve_bracket applied to the kernel's own raw scores and winners.  S = 149 draws: N is ragged."""
    S, seed = 149, 2000 + R * 100 + T_tab + F
    s, fx, hs, as_, tab, br = _case(model, S, T_tab, grouped, F, seed, best=best)
    k = _run(model, s, fx, hs, as_, tab, br, 15, R, seed)
    o = tournament.simulate_tournament(model, s, fx if F else None, hs, as_, tab, br, 15, R, seed)
    assert k["invalid"][0] == 0 and o["invalid"] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    gdiff = (kh != o["home"]) | (ka != o["away"])
    assert not (gdiff & ~(o["margin"] < 1e-5)).any(), np.argwhere(gdiff & ~(o["margin"] < 1e-5))[:5]
    kk = {x: k[x].astype(np.int64) for x in ("ko_scores", "ko_winners", "ko_entrants")}
    # ties whose entrants agree: their scores / winners agree unless an oracle margin is at rounding level
    same_ent = (kk["ko_entrants"] == o["ko_entrants"]).all(axis=2)
    diff = (kk["ko_scores"] != o["ko_scores"]).any(axis=2) | (kk["ko_winners"] != o["ko_winners"])
    small_ko = (o["ko_margin"] < 1e-5) | (o["decider_margin"] < 1e-5)
    assert not (diff & same_ent & ~small_ko).any(), np.argwhere(diff & same_ent & ~small_ko)[:5]
    assert gdiff.sum() <= max(1, 1e-3 * gdiff.size) and (diff | ~same_ent).sum() <= max(2, 1e-3 * diff.size)
    ent = kk["ko_entrants"]
    through = kk["ko_winners"] == ent[:, :, 0]
    r = tournament.resolve_bracket(tab, hs, as_, br, kh, ka, o["keys"], kk["ko_scores"][:, :, 0],
                                   kk["ko_scores"][:, :, 1], through)
    for key in ("ko_entrants", "ko_winners", "reach_counts", "win_counts", "positions", "position_counts",
                "points_counts"):
        np.testing.assert_array_equal(k[key], r[key], err_msg=key)
    K = len(br["round"])
    assert k["reach_counts"].sum() == 2 * K * S * R and k["win_counts"].sum() == K * S * R


def test_group_stage_is_bitwise_simulate_table():
    """Same seed and fixtures as bplx_simulate_table: positions, scores and both histograms are the same bits."""
    from bpl_next_b200 import simulate_table

    s, fx, hs, as_, tab, br = _case("neutral_wc", 150, 16, True, 60, seed=7, best=True)
    k = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 5, seed=17)
    g = simulate_table("neutral_wc", _dev(s), _dev(dict(fx, home_slot=hs, away_slot=as_)), _dev_table(tab), 15, 5, 17,
                       want_positions=True, want_scores=True)
    assert k["invalid"][0] == 0 and int(g["invalid"].item()) == 0
    for key in ("position_counts", "points_counts", "positions", "scores"):
        np.testing.assert_array_equal(k[key], g[key].cpu().numpy(), err_msg=key)


def test_draw_ranges_and_seeds():
    s, fx, hs, as_, tab, br = _case("neutral_wc", 50, 16, True, 40, seed=5, best=True)
    full = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=99)
    parts = [_run("neutral_wc", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, br, 15, 3, seed=99,
                  first_draw=lo) for lo, hi in ((0, 17), (17, 50))]
    for key in ("position_counts", "points_counts", "reach_counts", "win_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key])
    for key in ("positions", "scores", "ko_entrants", "ko_scores", "ko_winners"):
        np.testing.assert_array_equal(full[key], np.concatenate([p[key] for p in parts]))
    again = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=99)
    for key in ("reach_counts", "win_counts", "ko_winners", "ko_scores"):
        np.testing.assert_array_equal(full[key], again[key])
    other = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=100)
    assert not np.array_equal(full["ko_scores"], other["ko_scores"])
    noraw = _run("neutral_wc", s, fx, hs, as_, tab, br, 15, 3, seed=99, raw=False)
    for key in ("reach_counts", "win_counts", "position_counts"):
        np.testing.assert_array_equal(full[key], noraw[key])


def test_one_neutral_tie_against_the_per_draw_grids():
    """One neutral WC tie, N = 2^22: P(home advances) within 5 sigma of the mean over draws of hw_s / (hw_s + aw_s),
    and every score cell within 5 sigma of score_grid of the same draws."""
    from bpl_next_b200 import score_grid

    S, R = 64, 65536
    N = S * R
    s = make_samples("neutral_wc", S, 5, 4, seed=21)
    tab = season.build_table(["S0", "S1"])
    tab["num_points_bins"], tab["num_positions"] = 1, 2
    br = season.build_bracket(tab, [{"id": "f", "round": "F", "home": ("team", "S0"), "away": ("team", "S1"),
                                     "neutral_venue": 1}])
    br["slot_team"] = np.array([3, 1], np.uint16)
    br["slot_conf"] = np.array([2, 0], np.uint8)
    k = _run("neutral_wc", s, {}, np.zeros(0, np.uint8), np.zeros(0, np.uint8), tab, br, 15, R, seed=3)
    assert k["invalid"][0] == 0
    fx = {"home_team": np.array([3], np.uint16), "away_team": np.array([1], np.uint16),
          "home_conf": np.array([2], np.uint8), "away_conf": np.array([0], np.uint8),
          "neutral_venue": np.array([1], np.uint8)}
    lh, la = op.expected_goals("neutral_wc", s, fx["home_team"], fx["away_team"], home_conf=fx["home_conf"],
                               away_conf=fx["away_conf"], neutral_venue=fx["neutral_venue"])
    hw, aw = tournament.win_masses(lh[:, 0], la[:, 0], s["corr_coef"].astype(np.float64), 15)
    p = (hw / (hw + aw)).mean()
    share = (k["ko_winners"][:, 0] == 0).mean()
    assert abs(share - p) <= 5 * np.sqrt(p * (1 - p) / N), (share, p)
    grid, _ = score_grid("neutral_wc", _dev(s), _dev(fx), 15)
    pc = grid[0].double().cpu().numpy()
    counts = np.bincount(k["ko_scores"][:, 0, 0].astype(np.int64) * 16 + k["ko_scores"][:, 0, 1],
                         minlength=256).reshape(16, 16)
    assert (np.abs(counts - N * pc) <= 5 * np.sqrt(N * pc * (1 - pc)) + 1).all()


def test_knockout_only_bracket():
    """Eight teams, F = 0, SLOT entrants: sum_t win_counts of round r = (ties in r) N, champion probabilities sum to 1,
    every entrant reaches round 0."""
    s, fx, hs, as_, tab, br = _case("dixon_coles", 64, 8, False, 0, seed=51)
    N = 64 * 32
    k = _run("dixon_coles", s, fx, hs, as_, tab, br, 15, 32, seed=4, raw=False)
    assert k["invalid"][0] == 0
    ties_per_round = np.bincount(br["round"], minlength=br["num_rounds"])
    np.testing.assert_array_equal(k["win_counts"].sum(axis=0), ties_per_round * N)
    np.testing.assert_array_equal(k["reach_counts"][:, 0], N)
    pr = season.bracket_probabilities(br, k["reach_counts"], k["win_counts"], N)
    assert abs(pr["champion_proba"].sum() - 1.0) < 1e-12
    assert k["position_counts"].sum() == N * 8


def _wc_predictor(S=256, seed=61):
    """A NeutralWC predictor with synthetic posterior draws for 60 teams in 6 confederations."""
    from bpl_next_b200 import NeutralDixonColesMatchPredictorWC

    T, Cf = 60, 6
    s = make_samples("neutral_wc", S, T, Cf, seed=seed)
    m = NeutralDixonColesMatchPredictorWC()
    m.teams = [f"T{i:02d}" for i in range(T)]
    m._teams_dict = {t: i for i, t in enumerate(m.teams)}
    m.conferences = [f"C{i}" for i in range(Cf)]
    m._conferences_dict = {c: i for i, c in enumerate(m.conferences)}
    for k, v in s.items():
        setattr(m, k, v)
    return m


def _world_cup_48():
    """12 groups of four (round robins at neutral venues), the 8 best thirds through a generated complete 495-row
    allocation, a round of 32, 16, QF, SF, third-place match and final: 32 ties."""
    teams = [f"T{i:02d}" for i in range(48)]
    L = [chr(65 + g) for g in range(12)]
    groups = {t: L[i // 4] for i, t in enumerate(teams)}
    conf = {t: f"C{i % 6}" for i, t in enumerate(teams)}
    pairs = [(teams[4 * g + i], teams[4 * g + j]) for g in range(12) for i in range(4) for j in range(i + 1, 4)]
    fx = {"home_team": [a for a, _ in pairs], "away_team": [b for _, b in pairs],
          "home_conf": [conf[a] for a, _ in pairs], "away_conf": [conf[b] for _, b in pairs],
          "neutral_venue": [1] * len(pairs)}
    ent = [("group", g, 0) for g in L] + [("group", g, 1) for g in L] + [("best", j) for j in range(8)]
    ties = _knockout(ent, neutral=[1])
    for t in ties:
        t["round"] = {"r0": "R32", "r1": "R16", "r2": "QF", "r3": "SF", "r4": "F"}.get(t["round"], t["round"])
    best = {"position": 2, "count": 8, "allocation": _alloc(L, 8)}
    return teams, groups, fx, ties, best


def test_world_cup_48_end_to_end(monkeypatch):
    from bpl_next_b200 import DynamicNeutralDixonColesMatchPredictor, predictors

    m = _wc_predictor()
    teams, groups, fx, ties, best = _world_cup_48()
    assert len(ties) == 32 and len(best["allocation"]) == 495
    res = m.simulate_tournament(fx, ties, groups=groups, best=best, num_sims_per_draw=8, random_state=9)
    N = res["num_simulations"]
    assert N == 256 * 8 and res["rounds"] == ["R32", "R16", "QF", "SF", "third", "F"]
    assert res["reach_proba"].shape == (48, 6)
    np.testing.assert_allclose(res["reach_proba"][:, 0].sum(), 32.0, rtol=0, atol=1e-9)
    np.testing.assert_allclose(res["champion_proba"].sum(), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(res["reach_proba"][:, 5].sum(), 2.0, rtol=0, atol=1e-9)
    tab = m.simulate_table(fx, groups=groups, num_sims_per_draw=8, random_state=9)
    np.testing.assert_array_equal(res["position_proba"], tab["position_proba"])
    # a third (position 2) reaches the round of 32 only as one of the 8 best: 8 of the 12 thirds per simulation
    thirds = res["position_proba"][:, 2]
    assert np.all(res["reach_proba"][:, 0] <= res["position_proba"][:, :3].sum(axis=1) + 1e-12)
    assert thirds.sum() == pytest.approx(12.0)
    monkeypatch.setattr(predictors, "SIM_OUTPUT_BYTES", 8 * (48 + 2 * 72 + 5 * 32) * 100)  # ranges of 100 draws
    raw = m.simulate_tournament(fx, ties, groups=groups, best=best, num_sims_per_draw=8, random_state=9,
                                return_simulations=True)
    for key in ("position_proba", "points_proba", "reach_proba", "win_proba", "champion_proba"):
        np.testing.assert_array_equal(res[key], raw[key])
    assert raw["ko_winners"].shape == (N, 32) and raw["ko_entrants"].shape == (N, 32, 2)
    champ = np.bincount(raw["ko_winners"][:, -1], minlength=48) / N
    np.testing.assert_array_equal(champ, res["champion_proba"])
    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().simulate_tournament(fx, ties)


def _raw_call(model, s, tab, br, R=2, slot_team=None):
    """bplx_simulate_tournament with F = 0, called directly (no Python-side checks); returns the status."""
    from bpl_next_b200 import problem

    lib = _abi.lib()
    keep = []
    ptr = problem._device_ptr_fn(keep)
    st = problem._samples_struct(model, _dev(s), ptr)
    ft = _abi.Fixtures()
    t = problem._table_struct(dict(_dev_table(tab), num_points_bins=1, points_win=3, points_draw=1), ptr)
    b = problem._bracket_struct(dict(br, slot_team=br["slot_team"] if slot_team is None else slot_team), keep)
    K, nr = b.num_ties, max(b.num_rounds, 1)
    cnt = [torch.empty(64 * 64, dtype=torch.int64, device="cuda") for _ in range(5)]
    ws = torch.empty(1 << 22, dtype=torch.uint8, device="cuda")
    rc = lib.bplx_simulate_tournament(C.byref(st), C.byref(ft), None, None, C.byref(t), C.byref(b), 15, R, 1, 0,
                                      ptr(cnt[0]), ptr(cnt[1]), ptr(cnt[2]), ptr(cnt[3]), None, None, None, None, None,
                                      ptr(cnt[4]), ptr(ws), ws.numel(), None)
    torch.cuda.synchronize()
    return rc


def test_refusals():
    s, fx, hs, as_, tab, br = _case("dixon_coles", 8, 8, False, 0, seed=71)
    assert _raw_call("dixon_coles", s, tab, br) == _abi.OK
    with pytest.raises(_abi.BplxError):
        _run("dynamic", s, fx, hs, as_, tab, br, 15, 2, seed=1)
    # more than 64 ties
    many = {k: (np.resize(v, (65,) + np.shape(v)[1:]) if k in ("kind", "arg0", "arg1", "round", "neutral_venue")
                else v) for k, v in br.items()}
    many["kind"][:] = _abi.ENTRANT_SLOT
    many["round"][:] = 0
    assert _raw_call("dixon_coles", s, tab, many) == _abi.E_UNSUPPORTED
    # a forward reference and a BEST beyond best_count
    fwd = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in br.items()}
    fwd["kind"][0, 0], fwd["arg0"][0, 0] = _abi.ENTRANT_WINNER, 3
    assert _raw_call("dixon_coles", s, tab, fwd) == _abi.E_INVALID
    fwd["kind"][0, 0], fwd["arg0"][0, 0] = _abi.ENTRANT_BEST, 0
    assert _raw_call("dixon_coles", s, tab, fwd) == _abi.E_INVALID
    # a bad allocation row: a group outside its mask
    s4, fx4, hs4, as4, tab4, br4 = _case("dixon_coles", 8, 16, True, 20, seed=72, best=True)
    bad = dict(br4, best_alloc=br4["best_alloc"].copy())
    row = next(m for m in range(16) if bin(m).count("1") == 2)
    bad["best_alloc"][row] = [next(g for g in range(4) if not (row >> g) & 1), 0xFF]
    with pytest.raises(_abi.BplxError, match="allocation row"):
        _run("dixon_coles", s4, fx4, hs4, as4, tab4, bad, 15, 2, seed=1)
    # slot_team outside the model
    assert _raw_call("dixon_coles", s, tab, br, slot_team=np.full(8, 99, np.uint16)) == _abi.E_INVALID
    # N >= 2^31 in one call
    assert _raw_call("dixon_coles", s, tab, br, R=2 ** 28) == _abi.E_UNSUPPORTED
