"""Match importance on the GPU: the conditional kernel's counts replayed to the bit by oracle/conditional.py for all four
models, both ranking rules, one table and groups, R in {1, 64}, Kc and E at 1 and 64 and ragged N; a full 20-team
season at size against the host counts of its raw rows; every other output unchanged; draw ranges and key groups; a
hand-checkable two-team case; refusals; the predictor end to end."""
import ctypes as C

import numpy as np
import pytest
import torch

from bpl_next_b200 import _abi, problem, season
from oracle import conditional as oc
from oracle import head_to_head as h2h
from oracle import simulate as osim
from tests import test_head_to_head_gpu as th2h
from tests import test_simulate_gpu as tsim
from tests.test_score_grid_gpu import make_samples

pytestmark = pytest.mark.gpu

MODELS = ["dixon_coles", "extended", "neutral", "neutral_wc"]
RULES = ["goal_difference", "head_to_head"]


def _conditions(tab, F, Kc, E, seed):
    """Kc random key fixtures (sorted) and E random events (a slot and a non-empty set of its group's positions)."""
    rng = np.random.default_rng(seed)
    T = len(tab["start_points"])
    group = np.zeros(T, np.int64) if tab.get("group") is None else np.asarray(tab["group"], np.int64)
    size = np.bincount(group)[group]
    slots = rng.integers(0, T, E)
    masks = [int(rng.integers(1, 1 << int(size[t]))) if size[t] < 63 else int(rng.integers(1, 1 << 62)) for t in slots]
    return {"key_fixture": np.sort(rng.permutation(F)[:Kc]).astype(np.int32), "event_slot": slots.astype(np.uint8),
            "event_positions": np.asarray(masks, np.uint64)}


def _run(model, s, fx, hs, as_, tab, G, R, seed, cond=None, first_draw=0, raw=True):
    out = problem.simulate_table(model, tsim._dev(s), tsim._dev(dict(fx, home_slot=hs, away_slot=as_)),
                                 th2h._dev_table(tab), G, R, seed, first_draw=first_draw, want_positions=raw,
                                 want_scores=raw, conditions=cond)
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def _rank(tab, hs, as_, kh, ka, keys):
    if tab.get("tiebreak", "goal_difference") == "goal_difference":
        return osim.rank_scores(tab, hs, as_, kh, ka, keys)["positions"]
    return h2h.rank_scores(tab, hs, as_, kh, ka, keys, played_h2h=tab.get("played_h2h"))["positions"]


def _check_identities(k, cond):
    pc = k["position_counts"]
    n = int(pc[0].sum())
    np.testing.assert_array_equal(k["outcome_counts"].sum(axis=1), n)
    for e, (t, m) in enumerate(zip(cond["event_slot"], cond["event_positions"])):
        want = sum(int(pc[t, p]) for p in range(pc.shape[1]) if (int(m) >> p) & 1)
        np.testing.assert_array_equal(k["conditional_counts"][:, :, e].sum(axis=1), want)


# (R, T_tab, grouped, F, Kc, E): N = S R with S = 149 (R = 1) or 37 (R = 64), neither a multiple of 128
REPLAY = [(1, 20, False, 70, 1, 64), (64, 20, True, 60, 40, 1), (1, 64, True, 100, 64, 64), (64, 12, False, 64, 64, 9)]


@pytest.mark.parametrize("rule", RULES)
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("R,T_tab,grouped,F,Kc,E", REPLAY)
def test_exact_replay(model, rule, R, T_tab, grouped, F, Kc, E):
    """The kernel's counts equal oracle/conditional.py's counts of the kernel's own raw rows, integer for integer (its
    scores equal the oracle's except at rounding-level margins, and its positions are the oracle's ranking of them, as
    test_simulate_gpu / test_head_to_head_gpu check); where no score differs, they equal the full replay's counts."""
    S, seed = (149 if R == 1 else 37), 5000 + R + T_tab + F
    s, fx, hs, as_, tab = tsim._case(model, S, T_tab, grouped, F, seed)
    if rule == "head_to_head":
        tab = th2h._h2h(tab, th2h._played(T_tab, seed))
    cond = _conditions(tab, F, Kc, E, seed)
    k = _run(model, s, fx, hs, as_, tab, 15, R, seed, cond)
    assert k["invalid"][0] == 0
    kh, ka = k["scores"][:, :, 0].astype(np.int64), k["scores"][:, :, 1].astype(np.int64)
    keys = osim.philox_words(s, R, seed, 0, 2 * F + T_tab)[0][:, 2 * F:].astype(np.int64)
    pos = _rank(tab, hs, as_, kh, ka, keys)
    np.testing.assert_array_equal(k["positions"], pos)
    want = oc.counts(kh, ka, pos, np.ones(len(kh), bool), cond["key_fixture"], cond["event_slot"],
                     cond["event_positions"])
    np.testing.assert_array_equal(k["outcome_counts"], want[0])
    np.testing.assert_array_equal(k["conditional_counts"], want[1])
    _check_identities(k, cond)
    o = oc.simulate(model, s, fx, hs, as_, tab, 15, R, seed, cond, tiebreak=rule, played_h2h=tab.get("played_h2h"))
    if not ((kh != o["home"]) | (ka != o["away"])).any():
        np.testing.assert_array_equal(k["outcome_counts"], o["outcome_counts"])
        np.testing.assert_array_equal(k["conditional_counts"], o["conditional_counts"])


def _league(S, seed=7):
    """A 20-team double round robin (380 fixtures) on DixonColes draws for 20 teams."""
    s = make_samples("dixon_coles", S, 20, 4, seed=seed)
    names = [f"T{i:02d}" for i in range(20)]
    tab = season.build_table(names)
    pairs = [(i, j) for i in range(20) for j in range(20) if i != j]
    hs, as_ = season.fixture_slots(tab, [names[i] for i, _ in pairs], [names[j] for _, j in pairs])
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16)}
    return s, fx, hs, as_, tab


def test_at_size_against_the_raw_rows():
    """F = 380, S = 16,384 x R = 64 (2^20 seasons), Kc = E = 64: the counts recomputed on the host from the raw
    positions and scores equal the kernel's, bit for bit."""
    s, fx, hs, as_, tab = _league(16384)
    cond = _conditions(tab, 380, 64, 64, seed=3)
    k = _run("dixon_coles", s, fx, hs, as_, tab, 15, 64, 11, cond)
    assert k["invalid"][0] == 0
    want = oc.counts(k["scores"][:, :, 0], k["scores"][:, :, 1], k["positions"], np.ones(len(k["positions"]), bool),
                     cond["key_fixture"], cond["event_slot"], cond["event_positions"])
    np.testing.assert_array_equal(k["outcome_counts"], want[0])
    np.testing.assert_array_equal(k["conditional_counts"], want[1])
    _check_identities(k, cond)


@pytest.mark.parametrize("rule", RULES)
def test_nothing_else_moves(rule):
    s, fx, hs, as_, tab = tsim._case("neutral_wc", 61, 20, True, 60, seed=11)
    if rule == "head_to_head":
        tab = th2h._h2h(tab, th2h._played(20, 4))
    plain = _run("neutral_wc", s, fx, hs, as_, tab, 15, 5, 7)
    with_c = _run("neutral_wc", s, fx, hs, as_, tab, 15, 5, 7, _conditions(tab, 60, 64, 64, seed=1))
    for key in ("position_counts", "points_counts", "invalid", "positions", "scores"):
        np.testing.assert_array_equal(plain[key], with_c[key], err_msg=key)


def test_draw_ranges_key_groups_and_identities():
    s, fx, hs, as_, tab = tsim._case("neutral", 50, 12, True, 100, seed=5)
    cond = _conditions(tab, 100, 30, 20, seed=8)
    full = _run("neutral", s, fx, hs, as_, tab, 15, 3, 99, cond, raw=False)
    parts = [_run("neutral", {k: v[lo:hi] for k, v in s.items()}, fx, hs, as_, tab, 15, 3, 99, cond, first_draw=lo,
                  raw=False) for lo, hi in ((0, 17), (17, 50))]
    for key in ("outcome_counts", "conditional_counts", "position_counts"):
        np.testing.assert_array_equal(full[key], parts[0][key] + parts[1][key], err_msg=key)
    _check_identities(full, cond)
    # all 100 fixtures as keys, in the builder's groups of at most 64, equal one run per fixture
    events = {f"e{e}": (tab["teams"][int(t)], [p for p in range(4) if (int(m) >> p) & 1])
              for e, (t, m) in enumerate(zip(cond["event_slot"], cond["event_positions"]))}
    built = season.build_conditions(tab, 100, list(range(99, -1, -1)), events)
    assert len(built["groups"]) == 2
    oc_, cc = np.zeros((100, 3), np.int64), np.zeros((100, 3, 20), np.int64)
    for g in built["groups"]:
        r = _run("neutral", s, fx, hs, as_, tab, 15, 3, 99, dict(g, event_slot=built["event_slot"],
                                                                 event_positions=built["event_positions"]), raw=False)
        oc_[g["rows"]], cc[g["rows"]] = r["outcome_counts"], r["conditional_counts"]
    for f in range(100):
        one = _run("neutral", s, fx, hs, as_, tab, 15, 3, 99, dict(cond, key_fixture=np.array([f], np.int32)),
                   raw=False)
        np.testing.assert_array_equal(oc_[99 - f], one["outcome_counts"][0])
        np.testing.assert_array_equal(cc[99 - f], one["conditional_counts"][0])


def test_two_teams_one_fixture_by_hand():
    """Slots A (0) and B (1), one fixture A v B, no played results: P(A first | A wins) = 1, P(A first | B wins) = 0,
    and the draw row counts the drawn seasons whose tie-break key sends A first (key_A > key_B, or equal keys)."""
    s = make_samples("dixon_coles", 200, 2, 4, seed=9)
    tab = season.build_table(["A", "B"])
    hs, as_ = season.fixture_slots(tab, ["A"], ["B"])
    fx = {"home_team": np.array([0], np.uint16), "away_team": np.array([1], np.uint16)}
    cond = {"key_fixture": np.array([0], np.int32), "event_slot": np.array([0], np.uint8),
            "event_positions": np.array([1], np.uint64)}
    k = _run("dixon_coles", s, fx, hs, as_, tab, 15, 50, 3, cond)
    o, c = k["outcome_counts"][0], k["conditional_counts"][0, :, 0]
    assert o.min() > 0 and o.sum() == 200 * 50
    assert c[0] == o[0] and c[2] == 0
    words = osim.philox_words(s, 50, 3, 0, 4)[0].astype(np.int64)
    drawn = k["scores"][:, 0, 0] == k["scores"][:, 0, 1]
    assert c[1] == int((drawn & (words[:, 2] >= words[:, 3])).sum())
    assert 0 < c[1] < o[1]


def _raw(cond_struct, outcome=True, cond_out=True):
    """bplx_simulate_table_conditional called directly on a 6-slot table with 15 fixtures; returns the status."""
    s, fx, hs, as_, tab = tsim._case("dixon_coles", 8, 6, False, 15, seed=43)
    keep = []
    ptr = problem._device_ptr_fn(keep)
    lib = _abi.lib()
    st = problem._samples_struct("dixon_coles", tsim._dev(s), ptr)
    ft = problem._fixtures_struct(tsim._dev(fx), ptr)
    t = problem._table_struct(tsim._dev_table(tab), ptr)
    slots = tsim._dev({"h": hs, "a": as_})
    i64 = dict(dtype=torch.int64, device="cuda")
    pc, bc, inv = torch.empty((6, 6), **i64), torch.empty((6, t.num_points_bins), **i64), torch.empty(1, **i64)
    o, c = torch.empty((64, 3), **i64), torch.empty((64, 3, 64), **i64)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    rc = lib.bplx_simulate_table_conditional(
        C.byref(st), C.byref(ft), ptr(slots["h"]), ptr(slots["a"]), C.byref(t), None,
        None if cond_struct is None else C.byref(cond_struct), 15, 2, 1, 0, ptr(pc), ptr(bc),
        ptr(o) if outcome else None, ptr(c) if cond_out else None, None, None, ptr(inv), ptr(ws), ws.numel(), None)
    torch.cuda.synchronize()
    return rc


def test_refusals():
    def make(keys=(1, 4), slots=(0, 5), masks=(1, 7)):
        keep = []
        return problem._conditions_struct({"key_fixture": list(keys), "event_slot": list(slots),
                                           "event_positions": np.asarray(masks, np.uint64)}, keep), keep

    ok, keep = make()
    assert _raw(ok) == _abi.OK and _raw(None, False, False) == _abi.OK
    for bad in (make(keys=()), make(keys=range(65)), make(keys=(1, 15)), make(keys=(-1, 3)), make(keys=(4, 4)),
                make(keys=(5, 2)), make(slots=(), masks=()), make(slots=(0, 6)), make(masks=(0, 1)),
                make(masks=(1, 1 << 6)), make(slots=range(65), masks=[1] * 65)):
        assert _raw(bad[0]) == _abi.E_INVALID, _abi.lib().bplx_last_error()
    assert _raw(ok, outcome=False) == _abi.E_INVALID
    assert _raw(ok, cond_out=False) == _abi.E_INVALID
    s, fx, hs, as_, tab = tsim._case("dixon_coles", 8, 4, False, 6, seed=43)
    with pytest.raises(_abi.BplxError):
        _run("dynamic", s, fx, hs, as_, tab, 15, 2, 1, _conditions(tab, 6, 2, 2, seed=1))


def test_end_to_end_predictors():
    """A DixonColes league, a NeutralWC group stage and the dynamic predictor at a gameweek through simulate_table."""
    from bpl_next_b200 import DixonColesMatchPredictor
    from tests import test_dynamic_predict_gpu as tdyn
    from tests import test_tournament_gpu as ttour

    s, fx, hs, as_, tab = _league(256)
    m = DixonColesMatchPredictor()
    m.teams = np.array(tab["teams"])
    m._teams_dict = {t: i for i, t in enumerate(m.teams)}
    m.attack, m.defence, m.home_advantage, m.corr_coef = s["attack"], s["defence"], s["home_advantage"], s["corr_coef"]
    names = list(m.teams)
    fixtures = {"home_team": [names[i] for i in hs], "away_team": [names[i] for i in as_]}
    events = {f"{t} title": (t, 0) for t in names} | {f"{t} down": (t, (17, 18, 19)) for t in names}
    keys = list(range(379, 279, -1))  # 100 key fixtures: two groups
    res = m.simulate_table(fixtures, num_sims_per_draw=8, random_state=4, key_fixtures=keys, events=events)
    plain = m.simulate_table(fixtures, num_sims_per_draw=8, random_state=4)
    np.testing.assert_array_equal(res["position_proba"], plain["position_proba"])
    assert res["key_fixtures"] == keys and res["events"] == list(events)
    N = res["num_simulations"]
    np.testing.assert_array_equal(res["outcome_counts"].sum(axis=1), N)
    np.testing.assert_allclose(res["event_proba"][:20], res["position_proba"][:, 0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res["event_proba"][20:], res["position_proba"][:, 17:].sum(axis=1), rtol=0, atol=1e-12)
    cp = res["conditional_proba"]
    np.testing.assert_allclose(np.nansum(cp * res["outcome_proba"][:, :, None], axis=1),
                               np.broadcast_to(res["event_proba"], (100, 40)), rtol=0, atol=1e-12)
    assert (res["importance"] >= 0).all() and res["importance"].max() > 0
    # the last key fixture alone gives its row
    one = m.simulate_table(fixtures, num_sims_per_draw=8, random_state=4, key_fixtures=[keys[-1]], events=events)
    np.testing.assert_array_equal(one["conditional_counts"][0], res["conditional_counts"][-1])
    with pytest.raises(ValueError, match="both or neither"):
        m.simulate_table(fixtures, key_fixtures=[0])
    raw = m.simulate_table(fixtures, num_sims_per_draw=2, random_state=4, key_fixtures=[5], events={"x": ("T00", 0)},
                           return_simulations=True)
    assert raw["positions"].shape == (256 * 2, 20)

    wc = ttour._wc_predictor(S=128)
    teams, groups, wfx, _, _ = ttour._world_cup_48()
    last = list(range(len(wfx["home_team"])))[-24:]
    ev = {f"{t} through": (t, (0, 1)) for t in teams}
    r = wc.simulate_table(wfx, groups=groups, num_sims_per_draw=4, random_state=2, key_fixtures=last, events=ev,
                          tiebreak="head_to_head")
    np.testing.assert_allclose(r["event_proba"], r["position_proba"][:, :2].sum(axis=1), rtol=0, atol=1e-12)
    assert r["conditional_proba"].shape == (24, 3, 48)

    p = tdyn._fake_fit()
    dfx = {"home_team": ["t0", "t1", "t2", "t3", "t4", "t5"], "away_team": ["t1", "t2", "t3", "t0", "t5", "t4"]}
    kw = dict(random_state=5, key_fixtures=[0, 3], events={"t0 top": ("t0", 0)})
    rp, rq = p.simulate_table(dfx, gameweek=1, **kw), p.at_gameweek(1, 5).simulate_table(dfx, **kw)
    for key in ("outcome_counts", "conditional_counts", "position_proba"):
        np.testing.assert_array_equal(rp[key], rq[key], err_msg=key)
