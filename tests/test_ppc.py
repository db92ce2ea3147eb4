"""CPU: posterior predictive checks -- the oracle's statistics against hand counts, the host summary module
(bpl_next_b200/ppc.py) against the oracle, the mid-p definition with ties, the dispersion, the C struct mirror, and the
predictor refusals that need no GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bpl_next_b200 import _abi
from bpl_next_b200 import ppc as bppc
from oracle import ppc as oppc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# four teams, five matches: 0-0, 2-1, 1-1, 0-3, 7-0 (the last one lumped into the "5+" row)
HT, AT = np.array([0, 1, 2, 3, 0]), np.array([1, 2, 3, 0, 2])
HG, AG = np.array([0, 2, 1, 0, 7]), np.array([0, 1, 1, 3, 0])


def test_oracle_statistics_by_hand():
    st = oppc.statistics(HT, AT, HG[None], AG[None], num_teams=5, score_bins=6, points=(3, 1))
    cells = np.zeros((6, 6), np.int64)
    for h, a in ((0, 0), (2, 1), (1, 1), (0, 3), (5, 0)):
        cells[h, a] += 1
    np.testing.assert_array_equal(st["score_counts"][0], cells)
    np.testing.assert_array_equal(st["outcome_counts"][0], [2, 2, 1])
    np.testing.assert_array_equal(st["goals"][0], [10, 5])
    assert st["total_goals_sq"][0] == 0 + 9 + 4 + 9 + 49
    # team 0: 0-0 home (1 pt), 3-0 away win at team 3 (3 pts), 7-0 home win (3 pts); team 4 never plays
    np.testing.assert_array_equal(st["team_points"][0], [7, 4, 1, 1, 0])
    np.testing.assert_array_equal(st["team_goals_for"][0], [0 + 3 + 7, 0 + 2, 1 + 1 + 0, 1 + 0, 0])
    np.testing.assert_array_equal(st["team_goals_against"][0], [0 + 0 + 0, 0 + 1, 2 + 1 + 7, 1 + 3, 0])
    # two bins: "0" and "1+"; points (2, 1)
    st2 = oppc.statistics(HT, AT, HG[None], AG[None], num_teams=5, score_bins=2, points=(2, 1))
    np.testing.assert_array_equal(st2["score_counts"][0], [[1, 1], [1, 2]])
    np.testing.assert_array_equal(st2["team_points"][0], [5, 3, 1, 1, 0])


def test_host_statistics_equal_the_oracle():
    rng = np.random.default_rng(3)
    M, T = 400, 13
    ht = rng.integers(0, T, M)
    at = (ht + rng.integers(1, T, M)) % T
    hg, ag = rng.poisson(1.5, (7, M)), rng.poisson(1.1, (7, M))
    hg[0, :3] = 20  # above any score bin and any max_goals
    for B, pts in ((6, (3, 1)), (2, (2, 1)), (16, (1, 0))):
        o = oppc.statistics(ht, at, hg, ag, T, B, pts)
        for i in range(7):
            h = bppc.statistics(ht, at, hg[i], ag[i], T, B, pts)
            assert set(h) == set(bppc.STATISTICS)
            for k in bppc.STATISTICS:
                np.testing.assert_array_equal(h[k], o[k][i], err_msg=k)


def test_mid_p_with_ties():
    rep = np.array([[0, 5], [1, 5], [1, 6], [2, 7]])
    obs = np.array([1, 5])
    # element 0: one above, two tied -> (1 + 1) / 4; element 1: two above, two tied -> (2 + 1) / 4
    np.testing.assert_allclose(bppc.mid_p(rep, obs), [0.5, 0.75])
    np.testing.assert_allclose(oppc.mid_p(rep, obs), [0.5, 0.75])
    assert bppc.mid_p(np.zeros((9, 1)), np.zeros(1))[0] == 0.5  # every replicate equal: 0.5
    assert bppc.mid_p(np.arange(10)[:, None], np.array([-1]))[0] == 1.0
    assert bppc.mid_p(np.arange(10)[:, None], np.array([10]))[0] == 0.0


def test_dispersion():
    tot = np.array([0, 1, 2, 3, 4, 2])
    goals = np.array([tot.sum() - 3, 3])
    want = tot.var() / tot.mean()
    assert bppc.dispersion(goals, (tot ** 2).sum(), len(tot)) == pytest.approx(want, rel=1e-14)
    # per replicate: leading axes are kept
    d = bppc.dispersion(np.stack([goals, goals]), np.array([(tot ** 2).sum()] * 2), len(tot))
    np.testing.assert_allclose(d, [want, want], rtol=1e-14)
    # Poisson totals: close to 1
    x = np.random.default_rng(1).poisson(2.7, 200_000)
    assert bppc.dispersion(np.array([x.sum(), 0]), (x ** 2).sum(), len(x)) == pytest.approx(1.0, abs=0.02)


def test_summarize():
    rng = np.random.default_rng(5)
    M, T, N = 50, 6, 300
    ht = rng.integers(0, T - 1, M)  # team T - 1 never plays
    at = (ht + rng.integers(1, T - 1, M)) % (T - 1)
    hg, ag = rng.poisson(1.4, (N, M)), rng.poisson(1.2, (N, M))
    reps = oppc.statistics(ht, at, hg, ag, T)
    obs = bppc.statistics(ht, at, hg[0], ag[0], T)
    res = bppc.summarize(obs, reps, M)
    assert set(res) == set(bppc.STATISTICS) | {"total_goals_dispersion"}
    for k, v in res.items():
        assert set(v) == {"observed", "mean", "sd", "p_value"}
        r = np.asarray(reps[k]) if k in reps else bppc.dispersion(reps["goals"], reps["total_goals_sq"], M)
        np.testing.assert_allclose(v["mean"], r.mean(axis=0), rtol=1e-14)
        np.testing.assert_allclose(v["sd"], r.std(axis=0), rtol=1e-12)
        np.testing.assert_allclose(v["p_value"], oppc.mid_p(r, v["observed"]), rtol=0, atol=1e-15)
        assert v["p_value"].shape == np.shape(v["observed"])
    assert res["team_points"]["p_value"][T - 1] == 0.5
    assert res["total_goals_dispersion"]["observed"] == pytest.approx(
        bppc.dispersion(obs["goals"], obs["total_goals_sq"], M))


def test_output_struct_mirrors_the_header():
    src = open(os.path.join(ROOT, "include", "bplx.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} bplx_ppc_output;", src).group(1)
    fields = re.findall(r"\*\s*(\w+);", body)
    assert fields == [f for f, _ in _abi.PpcOutput._fields_]
    assert C.sizeof(_abi.PpcOutput) == 9 * 8
    assert fields[:7] == list(bppc.STATISTICS)
    assert re.search(r"int bplx_posterior_predictive\(", src)
    assert hasattr(_abi.lib(), "bplx_posterior_predictive")
    assert _abi.lib().bplx_posterior_predictive_workspace_bytes(None, None) == 0


def test_predictor_refusals_without_a_gpu():
    from bpl_next_b200 import DixonColesMatchPredictor, DynamicNeutralDixonColesMatchPredictor

    with pytest.raises(ValueError, match="not fitted"):
        DixonColesMatchPredictor().posterior_predictive_check()
    with pytest.raises(NotImplementedError):
        DynamicNeutralDixonColesMatchPredictor().posterior_predictive_check()
