"""CPU: randomised problems (sizes that force multi-stage streams, split list pieces, idle teams, duplicates, every
venue mix) -- the double-precision walk of the product's plan must equal the oracle for every split (1/2/4/8 CTAs)."""
import numpy as np
import pytest

from oracle import models as om
from tests import helpers as H

MODELS = ["dixon_coles", "extended", "neutral", "neutral_wc", "dynamic"]


def _random_problem(seed):
    rng = np.random.default_rng(seed)
    model = MODELS[seed % len(MODELS)]
    T = int(rng.integers(2, 40))
    M = int(rng.choice([1, 5, 60, 400, 2500]))
    kw = dict(T=T, M=M, low_scores=bool(rng.integers(0, 2)))
    if model != "dixon_coles":
        kw["K"] = int(rng.choice([0, 0, 1, 3]))
        kw["weighted"] = bool(rng.integers(0, 2))
    if model in ("neutral", "neutral_wc", "dynamic"):
        kw["neutral_frac"] = float(rng.choice([0.0, 0.3, 1.0]))
    if model == "neutral_wc":
        kw["Cf"] = int(rng.integers(1, 7))
        kw["multi_conf"] = bool(rng.integers(0, 2))
    if model == "dynamic":
        kw["Cf"] = int(rng.integers(1, 12))  # gameweeks
        kw.pop("weighted", None)
    if T < 3 and kw.get("K", 0):
        kw["K"] = 0  # a covariate column with two teams standardises to +-1: fine, but keep tiny cases simple
    return model, kw


@pytest.mark.parametrize("seed", range(40))
def test_random_problem_plan_matches_oracle(seed):
    model, kw = _random_problem(seed)
    arr = H.small_problem(model, seed=100 + seed, **kw)
    d = H.to_oracle(arr)
    D = om.num_params(model, arr.num_teams, arr.num_covariates, arr.num_conferences, arr.num_gameweeks)
    theta = H.random_theta(D, 2, seed=seed, radius=0.8)
    lp_o, g_o, cc_o = om.log_density_and_grad(d, theta)
    splits = (0,) if model == "dynamic" else (0, 1, 3)
    for si in splits:
        lp_p, g_p, cc_p = H.plancheck_eval(arr, theta, si)
        np.testing.assert_allclose(lp_p, lp_o, rtol=2e-7, err_msg=f"{model} {kw} split {1 << si}")
        np.testing.assert_allclose(cc_p, cc_o, rtol=1e-9, atol=1e-12)
        scale = np.abs(g_o).max(axis=1, keepdims=True)
        np.testing.assert_allclose(g_p / scale, g_o / scale, rtol=0, atol=3e-7)


GEOMETRY_WARPS = (1, 2, 3, 5, 7, 13, 24, 30)


@pytest.mark.parametrize("seed", range(0, 40, 2))
def test_plan_geometries_match_oracle(seed, monkeypatch):
    """The plan under forced geometries (BPLX_NWARPS warps per CTA, 512 / 1024-byte stages, phase 2 by (team, side) or
    by whole team; K1d: hyper table in shared memory or the workspace) walked in double == the oracle, for 1, 2 and 8 CTAs
    per chain group -- on the randomised problems and, for the covariate models, the same problem with K = 4 ... 16."""
    model, kw = _random_problem(seed)
    problems = [H.small_problem(model, seed=100 + seed, **kw)]
    if model != "dixon_coles" and kw["T"] >= 3:
        problems.append(H.small_problem(model, seed=100 + seed, **dict(kw, K=(4, 5, 8, 16)[seed % 4])))
    for arr in problems:
        d = H.to_oracle(arr)
        D = om.num_params(model, arr.num_teams, arr.num_covariates, arr.num_conferences, arr.num_gameweeks)
        theta = H.random_theta(D, 1, seed=seed, radius=0.8)
        lp_o, g_o, cc_o = om.log_density_and_grad(d, theta)
        scale = np.abs(g_o).max(axis=1, keepdims=True)
        if model == "dynamic":
            geoms = [dict(BPLX_NWARPS=W, BPLX_DYN_HYP_WS=h) for W in GEOMETRY_WARPS for h in (0, 1)]
            splits = (0,)
        else:
            geoms = [dict(BPLX_NWARPS=W, BPLX_STAGE=st, BPLX_NO_P2SPLIT=p2) for W in GEOMETRY_WARPS for st in (512, 1024)
                     for p2 in (None, 1)]
            splits = (0, 1, 3)
        for g in geoms:
            for k, v in g.items():
                if v is None:
                    monkeypatch.delenv(k, raising=False)
                else:
                    monkeypatch.setenv(k, str(v))
            for si in splits:
                lp_p, g_p, cc_p = H.plancheck_eval(arr, theta, si)
                msg = f"{model} K={arr.num_covariates} {g} split {1 << si}"
                np.testing.assert_allclose(lp_p, lp_o, rtol=2e-7, err_msg=msg)
                np.testing.assert_allclose(cc_p, cc_o, rtol=1e-9, atol=1e-12, err_msg=msg)
                np.testing.assert_allclose(g_p / scale, g_o / scale, rtol=0, atol=3e-7, err_msg=msg)
