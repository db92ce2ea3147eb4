"""GPU: K1 / K1d under plan geometries the planner does not pick by itself, on problems built to reach each path.

The testing switches (BPLX_NWARPS warps per CTA, BPLX_STAGE ring-stage bytes, BPLX_NO_P2SPLIT phase 2 by whole team,
BPLX_DYN_HYP_WS K1d's hyper table in the workspace) are read when the plan is built, so they are set before Problem().
Every call is checked against the float64 oracle with test_logdensity_gpu._check (which includes the per-component
criterion), and every case asserts from the plan statistics that it reached the path it is for."""
import ctypes as C

import numpy as np
import pytest

from tests import helpers as H
from tests.test_logdensity_gpu import _check

pytestmark = pytest.mark.gpu

K_STAGES = 2  # plan.h kStages


def _problems():
    """name -> MatchArrays."""
    out = {}
    out["few_team_ext"] = H.small_problem("extended", seed=3, T=5, M=200, K=3)  # phase 2 by (team, side)
    out["wc_conf"] = H.small_problem("neutral_wc", seed=3, T=13, M=400, K=2, multi_conf=True)  # P2 split refused
    out["long_dc"] = H.small_problem("dixon_coles", seed=4, T=30, M=2500)  # a W = 1 stream of many stages
    big = H.small_problem("neutral", seed=5, T=100, M=700, K=0)  # team 0 at home against 99 opponents: lists > 64
    big.home_team = big.home_team.copy()
    big.away_team = big.away_team.copy()
    big.home_team[:99] = 0
    big.away_team[:99] = np.arange(1, 100)
    out["long_list_neutral"] = big
    idle = H.small_problem("extended", seed=6, T=6, M=40, K=2)
    idle.num_teams = 9  # teams 6..8 never play
    idle.covariates = np.vstack([idle.covariates, np.zeros((3, 2), np.float32)])
    out["idle_ext"] = idle
    for model in ("extended", "neutral", "neutral_wc"):
        for K in (5, 16):
            out[f"{model}_K{K}"] = H.small_problem(model, seed=7, T=20, M=300, K=K)
    return out


PROBLEMS = _problems()


def _warp_stats(p, W):
    buf = (C.c_longlong * (W * 12))()
    n = p._lib.bplx_problem_warp_stats(p._h, buf, W * 12)
    return np.array(buf[:n], dtype=np.int64).reshape(-1, 2, 6)  # [warp][phase][pieces, ..., teams, stages]


class _Runner:
    """One theta batch per (problem, C); every call checked against the oracle."""

    def __init__(self, arr, C, seed=11, radius=0.8):
        from bpl_next_b200 import Problem
        self.arr = arr
        p = Problem(arr)
        self.theta = H.random_theta(p.D, C, seed=seed, radius=radius, dtype=np.float32)
        p.close()

    def run(self, what, minor=False):
        import torch
        from bpl_next_b200 import Problem
        p = Problem(self.arr)
        t = torch.from_numpy(self.theta).cuda()
        lp, grad, cc = p.logdensity(t.t().contiguous() if minor else t, chain_minor=minor)
        torch.cuda.synchronize()
        g = grad.t().contiguous() if minor else grad
        _check(self.arr, self.theta.astype(np.float64), lp.cpu().numpy(), g.cpu().numpy(), cc.cpu().numpy(), what)
        return p


def _geometry(monkeypatch, W=None, stage=None, no_p2=False, hyp_ws=None):
    for k, v in (("BPLX_NWARPS", W), ("BPLX_STAGE", stage), ("BPLX_DYN_HYP_WS", hyp_ws)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))
    if no_p2:
        monkeypatch.setenv("BPLX_NO_P2SPLIT", "1")
    else:
        monkeypatch.delenv("BPLX_NO_P2SPLIT", raising=False)


@pytest.mark.parametrize("name", ["few_team_ext", "wc_conf", "long_dc", "long_list_neutral", "idle_ext"])
def test_static_geometry_sweep(name, monkeypatch):
    """W in {1, 2, 5, 13, 24} x stage {512, 1024} x phase 2 dealt by (team, side) or by whole team."""
    arr = PROBLEMS[name]
    r = _Runner(arr, 45)
    smem = {}
    for W in (1, 2, 5, 13, 24):
        for stage in (512, 1024):
            for no_p2 in (False, True):
                _geometry(monkeypatch, W, stage, no_p2)
                p = r.run(f"{name} W={W} stage={stage} no_p2split={no_p2}")
                st = p.stats()
                assert st["warps"] == W
                smem[W, stage, no_p2] = st["smem_bytes"]
                ws = _warp_stats(p, W)
                assert ws.shape[0] == W
                if W == 1 and name == "long_dc":  # the single warp's streams wrap the two-stage ring many times
                    assert ws[0, 0, 5] > 4 * K_STAGES and ws[0, 1, 5] > K_STAGES, ws[0]
                if W == 24 and arr.num_teams < 24:  # more warps than teams with matches: idle warps
                    assert (ws[:, 0, 4] == 0).any() and (ws[:, 1, 4] == 0).any()
                if name == "long_list_neutral" and stage == 512:  # team 0's 99-entry home list is cut into pieces
                    p.close()
                    _geometry(monkeypatch, W, 1024, no_p2)
                    from bpl_next_b200 import Problem
                    q = Problem(arr)
                    assert ws[:, 0, 0].sum() > _warp_stats(q, W)[:, 0, 0].sum()
                    q.close()
                p.close()
    for W in (1, 2, 5, 13, 24):
        for stage in (512, 1024):
            if name == "few_team_ext" and W >= 13:  # phase 2 by (team, side): the side tables take shared memory
                assert smem[W, stage, False] > smem[W, stage, True], (W, stage)
            if name == "wc_conf":  # never with confederations
                assert smem[W, stage, False] == smem[W, stage, True], (W, stage)


@pytest.mark.parametrize("name", ["few_team_ext", "wc_conf", "idle_ext"])
@pytest.mark.parametrize("W", [1, 24])
def test_static_chain_counts_and_layouts(name, W, monkeypatch):
    """1, 31 and 45 chains (one lane, less than a warp, a ragged last CTA), chain-major and chain-minor."""
    _geometry(monkeypatch, W, 512)
    for Cn in (1, 31, 45):
        r = _Runner(PROBLEMS[name], Cn, seed=Cn)
        for minor in (False, True):
            r.run(f"{name} W={W} C={Cn} chain_minor={minor}", minor).close()


@pytest.mark.parametrize("split", [2, 8])
@pytest.mark.parametrize("W", [1, 5])
@pytest.mark.parametrize("name", ["few_team_ext", "wc_conf"])
def test_cluster_split_forced_warps(name, W, split, monkeypatch, bplx_env):
    bplx_env(BPLX_SPLIT=split)
    _geometry(monkeypatch, W, 512)
    for Cn in (45, 7):
        p = _Runner(PROBLEMS[name], Cn).run(f"{name} W={W} split={split} C={Cn}")
        assert p.stats()["warps"] == W
        p.close()


@pytest.mark.parametrize("W", [1, 13, 24])
def test_clip_forms_forced(W, monkeypatch):
    monkeypatch.setenv("BPLX_CLIP_FORMS", "3")
    _geometry(monkeypatch, W, 512)
    for name in ("few_team_ext", "idle_ext", "extended_K16"):
        _Runner(PROBLEMS[name], 45).run(f"{name} clip forms forced W={W}").close()


@pytest.mark.parametrize("name", [f"{m}_K{K}" for m in ("extended", "neutral", "neutral_wc") for K in (5, 16)])
def test_many_covariates(name, monkeypatch):
    """The prologue's loop over covariates k >= 4 (K = 5, 16), planner's choice and forced W."""
    r = _Runner(PROBLEMS[name], 45, radius=0.5)
    for W in (None, 1, 24):
        _geometry(monkeypatch, W, 512 if W else None)
        for minor in (False, True):
            p = r.run(f"{name} W={W} chain_minor={minor}", minor)
            if W:
                assert p.stats()["warps"] == W
            p.close()


DYN = {"dyn_T5": dict(Cf=4, T=5, M=90), "dyn_T23": dict(Cf=6, T=23, M=600, neutral_frac=0.2),
       "dyn_K5": dict(Cf=4, T=8, M=150, K=5), "dyn_K16": dict(Cf=4, T=20, M=300, K=16)}


@pytest.mark.parametrize("name", list(DYN))
def test_dynamic_geometry(name, monkeypatch):
    """K1d: W in {1, 3, 20} (one team per warp when T <= W) x hyper table in shared memory / in the workspace."""
    arr = H.small_problem("dynamic", seed=3, **DYN[name])
    T, G = arr.num_teams, arr.num_gameweeks
    r = _Runner(arr, 45, radius=0.5)
    for W in (1, 3, 20):
        smem = {}
        for hyp_ws in (0, 1):
            _geometry(monkeypatch, W, hyp_ws=hyp_ws)
            for minor in (False, True):
                p = r.run(f"{name} W={W} hyp_ws={hyp_ws} chain_minor={minor}", minor)
                st = p.stats()
                assert st["warps"] == min(W, T, 20)
                smem[hyp_ws] = st["smem_bytes"]
                p.close()
        assert smem[0] - smem[1] == G * 16 * 128  # the [G][16] hyper table moved out of shared memory


@pytest.mark.parametrize("W", [1, 24])
@pytest.mark.parametrize("model,kw", [("dixon_coles", dict()), ("extended", dict(weighted=True)),
                                      ("neutral", dict()), ("neutral_wc", dict(multi_conf=True, T=13, M=400))])
def test_likelihood_only_entry_point_forced_warps(model, kw, W, monkeypatch):
    from tests.test_logdensity_gpu import test_likelihood_only_entry_point
    _geometry(monkeypatch, W, 512)
    for minor in (False, True):
        test_likelihood_only_entry_point(model, kw, minor)
