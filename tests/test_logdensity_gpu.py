"""GPU parity: K1 (C ABI) vs the float64 oracle restatement of the reference models.

Tolerances are BASELINE.json's: log-density 1e-5 relative, gradient 1e-4 relative (float32)."""
import hashlib

import numpy as np
import pytest

from oracle import datasets, models as om
from tests import helpers as H

pytestmark = pytest.mark.gpu

LP_RTOL = 1e-5
GRAD_RTOL = 1e-4


_ORACLE = {}


def _check(arr, theta64, lp, grad, cc, what=""):
    """Against the float64 oracle: lp and corr_coef relative, the gradient scaled by its largest component, and every
    component within the per-component criterion (tests/helpers.py: CRIT_C 2^-24 sum |d term / d theta_i|)."""
    key = (id(arr), hashlib.sha1(np.ascontiguousarray(theta64).tobytes()).hexdigest())
    if key not in _ORACLE:  # (geometry sweeps check many calls on one problem and one theta)
        _ORACLE.clear()
        d = H.to_oracle(arr)
        _ORACLE[key] = (d, arr) + om.log_density_and_grad(d, theta64) + om.gradient_scale(d, theta64)
    d, _, lp_o, g_o, cc_o, kappa, lp_scale = _ORACLE[key]
    np.testing.assert_allclose(lp, lp_o, rtol=LP_RTOL)
    np.testing.assert_allclose(cc, cc_o, rtol=1e-4, atol=1e-6)
    scale = np.abs(g_o).max(axis=1, keepdims=True)
    err = np.abs(grad - g_o) / scale
    assert err.max() < GRAD_RTOL, f"max scaled gradient error {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"
    H.assert_criterion(d, theta64, lp, grad, what or arr.model, ref=(lp_o, g_o, kappa, lp_scale))


CASES = [
    ("dixon_coles", dict()),
    ("extended", dict(weighted=False)),
    ("extended", dict(weighted=True, K=3)),
    ("neutral", dict(K=2)),
    ("neutral", dict(neutral_frac=0.0)),
    ("neutral", dict(neutral_frac=1.0)),
    ("neutral_wc", dict()),
    ("neutral_wc", dict(multi_conf=True, K=2, T=13, M=400)),
    ("dynamic", dict(Cf=4, T=5, M=90)),
    ("dynamic", dict(Cf=3, T=6, M=120, K=2, neutral_frac=0.0)),
    ("dynamic", dict(Cf=5, T=4, M=40, as_written=True)),
    ("dynamic", dict(Cf=33, T=23, M=3000, neutral_frac=0.2)),
]


@pytest.mark.parametrize("model,kw", CASES)
@pytest.mark.parametrize("radius", [0.5, 2.0])
@pytest.mark.parametrize("chain_minor", [False, True])
def test_small_problems(model, kw, radius, chain_minor):
    import torch
    from bpl_next_b200 import Problem

    kw = dict(kw)
    as_written = kw.pop("as_written", False)
    arr = H.small_problem(model, seed=3, **kw)
    arr.as_written = as_written
    if model == "dynamic" and arr.num_gameweeks > 8 and radius > 1.0:
        pytest.skip("a 33-step walk of U(-2,2) steps overflows float32 rates (the reference's float32 path would too)")
    p = Problem(arr)
    C = 45  # not a multiple of 32: exercises the ragged last CTA
    theta = H.random_theta(p.D, C, seed=11, radius=radius, dtype=np.float32)
    t = torch.from_numpy(theta).cuda()
    if chain_minor:
        t = t.t().contiguous()
    lp, grad, cc = p.logdensity(t, chain_minor=chain_minor)
    torch.cuda.synchronize()
    g = grad.t().contiguous() if chain_minor else grad
    _check(arr, theta.astype(np.float64), lp.cpu().numpy(), g.cpu().numpy(), cc.cpu().numpy())


@pytest.mark.parametrize("model,eps", [("dixon_coles", None), ("extended", None), ("extended", 1.0),
                                       ("neutral", 0.5), ("neutral_wc", 0.2)])
def test_reference_fixtures_host_path(model, eps):
    """The reference's own test data (tests/conftest.py) through the host-buffer entry point."""
    from bpl_next_b200 import Problem

    td = {"dixon_coles": datasets.dummy_data, "extended": datasets.timed_dummy_data,
          "neutral": datasets.neutral_dummy_data, "neutral_wc": datasets.neutral_dummy_data}[model]()
    arr = H.from_training_data(model, td, epsilon=eps)
    p = Problem(arr)
    theta = H.random_theta(p.D, 64, seed=5, radius=1.0, dtype=np.float32)
    lp, grad, cc = p.logdensity_host(theta)
    _check(arr, theta.astype(np.float64), lp, grad, cc)


def test_survey_anchor():
    """SURVEY.md Appendix E anchor: theta_i = 0.3 sin(1+i) on conftest.dummy_data."""
    from bpl_next_b200 import Problem

    arr = H.from_training_data("dixon_coles", datasets.dummy_data())
    p = Problem(arr)
    theta = (0.3 * np.sin(1.0 + np.arange(45)))[None, :].astype(np.float32)
    lp, grad, cc = p.logdensity_host(theta)
    assert abs(lp[0] - (-1689.4267185765793)) < 1e-5 * 1689.5
    assert abs(cc[0] - 0.1544682575346078) < 1e-5
    assert abs(np.linalg.norm(grad[0]) - 883.2262464523642) < 1e-4 * 883.3


@pytest.mark.parametrize("cfg", ["config_2", "config_3", "config_4"])
def test_baseline_configs(cfg):
    """BASELINE.json configs at full match count, a handful of chains against the oracle."""
    import torch
    from bpl_next_b200 import Problem

    if cfg == "config_2":
        arr = H.from_training_data("extended", datasets.config_2(), epsilon=0.01)
    elif cfg == "config_4":
        arr = H.from_training_data("dynamic", datasets.config_4())
    else:
        arr = H.from_training_data("neutral_wc", datasets.config_3(), epsilon=0.1)
    p = Problem(arr)
    C = 40
    for radius in ((0.3, 0.8) if cfg == "config_4" else (0.3, 2.0)):  # a 30-step walk of U(-2,2) steps overflows float32 rates
        theta = H.random_theta(p.D, C, seed=21, radius=radius, dtype=np.float32)
        lp, grad, cc = p.logdensity(torch.from_numpy(theta).cuda())
        torch.cuda.synchronize()
        _check(arr, theta.astype(np.float64), lp.cpu().numpy(), grad.cpu().numpy(), cc.cpu().numpy())


def test_errors():
    from bpl_next_b200 import Problem, _abi

    arr = H.small_problem("dixon_coles")
    arr.home_team = arr.home_team.copy()
    arr.home_team[0] = 999
    with pytest.raises(_abi.BplxError) as e:
        Problem(arr)
    assert e.value.status == _abi.E_INVALID


def test_edge_cases():
    """One match, idle teams, zero weights / double-digit goals, single confederation with every venue neutral;
    1 chain and 31 chains (less than one warp of chains)."""
    import torch
    from bpl_next_b200 import Problem
    from tests.test_plan import _edge_cases

    for name, arr in _edge_cases():
        p = Problem(arr)
        for C in (1, 31):
            theta = H.random_theta(p.D, C, seed=17, radius=1.0, dtype=np.float32)
            for minor in (False, True):
                t = torch.from_numpy(theta).cuda()
                lp, grad, cc = p.logdensity(t.t().contiguous() if minor else t, chain_minor=minor)
                torch.cuda.synchronize()
                g = grad.t().contiguous() if minor else grad
                _check(arr, theta.astype(np.float64), lp.cpu().numpy(), g.cpu().numpy(), cc.cpu().numpy())
        p.close()


def test_results_are_bit_reproducible():
    """No atomics between warps on the gradient path: two calls on the same input give identical bits."""
    import torch
    from bpl_next_b200 import Problem

    arr = H.from_training_data("neutral_wc", datasets.neutral_dummy_data(), epsilon=0.2)
    p = Problem(arr)
    t = torch.from_numpy(H.random_theta(p.D, 96, seed=3, radius=1.5, dtype=np.float32)).cuda()
    a = [x.clone() for x in p.logdensity(t)]
    b = [x.clone() for x in p.logdensity(t)]
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("split", [1, 2, 4, 8])
@pytest.mark.parametrize("model,kw", [("extended", dict(weighted=True, K=3)), ("neutral_wc", dict(multi_conf=True, K=2, T=13, M=400)),
                                      ("dixon_coles", dict())])
def test_cluster_split(model, kw, split, bplx_env):
    """Few-chain mode: 1, 2, 4 or 8 CTAs (one thread-block cluster) share a group of chains; same numbers."""
    import torch
    from bpl_next_b200 import Problem

    bplx_env(BPLX_SPLIT=split)
    arr = H.small_problem(model, seed=3, **kw)
    p = Problem(arr)
    for C in (45, 7):
        theta = H.random_theta(p.D, C, seed=11, radius=1.0, dtype=np.float32)
        lp, grad, cc = p.logdensity(torch.from_numpy(theta).cuda())
        torch.cuda.synchronize()
        _check(arr, theta.astype(np.float64), lp.cpu().numpy(), grad.cpu().numpy(), cc.cpu().numpy())
    p.close()


@pytest.mark.parametrize("seed", range(0, 40, 3))
def test_random_problems(seed):
    """The randomised problems of tests/test_plan_random.py through the CUDA kernels (33 chains, both layouts)."""
    import torch
    from bpl_next_b200 import Problem
    from tests.test_plan_random import _random_problem

    model, kw = _random_problem(seed)
    arr = H.small_problem(model, seed=100 + seed, **kw)
    p = Problem(arr)
    theta = H.random_theta(p.D, 33, seed=seed, radius=0.8, dtype=np.float32)
    for minor in (False, True):
        t = torch.from_numpy(theta).cuda()
        lp, grad, cc = p.logdensity(t.t().contiguous() if minor else t, chain_minor=minor)
        torch.cuda.synchronize()
        g = grad.t().contiguous() if minor else grad
        _check(arr, theta.astype(np.float64), lp.cpu().numpy(), g.cpu().numpy(), cc.cpu().numpy())
    p.close()


@pytest.mark.parametrize("model,kw", [("dixon_coles", dict()), ("extended", dict(weighted=True, K=3))])
def test_clip_free_forms(model, kw, monkeypatch):
    """Models that clip their rates at 15 take a shorter form of the same arithmetic when no rate of a group of 32
    chains can reach the clip (prologue bound for phase 1, the reduced maxima for phase 2).  Near the mode (radius
    0.15: every rate far below 15) the short form must agree with the oracle, and it must give the same BITS as the
    clipping form: the same chains next to one far-out chain (which switches the whole group to the clipping form)."""
    import torch
    from bpl_next_b200 import Problem

    arr = H.small_problem(model, seed=3, **kw)
    p = Problem(arr)
    C = 64
    near = H.random_theta(p.D, C, seed=5, radius=0.15, dtype=np.float32)
    lp, grad, cc = [x.cpu().numpy() for x in p.logdensity(torch.from_numpy(near).cuda())]
    _check(arr, near.astype(np.float64), lp, grad, cc)
    mixed = near.copy()
    far = H.random_theta(p.D, 2, seed=9, radius=2.0, dtype=np.float32)
    mixed[7], mixed[40] = far[0], far[1]  # one far-out chain in each group of 32
    lp2, grad2, cc2 = [x.cpu().numpy() for x in p.logdensity(torch.from_numpy(mixed).cuda())]
    keep = np.ones(C, bool)
    keep[[7, 40]] = False
    assert np.array_equal(lp[keep], lp2[keep])
    assert np.array_equal(grad[keep], grad2[keep])
    assert np.array_equal(cc[keep], cc2[keep])
    _check(arr, mixed.astype(np.float64), lp2, grad2, cc2)
    p.close()
    # the same through the testing switch: phase 1 / phase 2 / both forced to the clipping form on the near batch
    for forms in ("1", "2", "3"):
        monkeypatch.setenv("BPLX_CLIP_FORMS", forms)
        q = Problem(arr)
        lp3, grad3, cc3 = [x.cpu().numpy() for x in q.logdensity(torch.from_numpy(near).cuda())]
        q.close()
        assert np.array_equal(lp, lp3) and np.array_equal(grad, grad3) and np.array_equal(cc, cc3), forms


def test_far_out_position_is_reproducible_and_rejectable():
    """A position the sampler visited in its first warm-up leapfrogs (|theta| up to 1,600: rates overflow float32 to inf
    and tie at the maximum).  The call must give the same bits every time -- the arg-max entry is chosen by atomicMin, not
    by the last finder -- and must not report a log-density of +inf (a sampler would accept it as the best point ever)."""
    import os
    import torch
    from bpl_next_b200 import Problem

    arr = H.from_training_data("dixon_coles", datasets.dummy_data())
    p = Problem(arr)
    far = np.load(os.path.join(os.path.dirname(__file__), "golden", "far_out_theta_dixon_coles.npy")).astype(np.float32)
    theta = H.random_theta(p.D, 64, seed=1, radius=1.0, dtype=np.float32)
    theta[5] = far
    theta[40] = far
    t = torch.from_numpy(theta).cuda()
    ref = [x.clone() for x in p.logdensity(t)]
    assert not torch.isposinf(ref[0]).any()
    for _ in range(20):
        out = p.logdensity(t)
        torch.cuda.synchronize()
        for a, b in zip(ref, out):
            assert torch.equal(torch.nan_to_num(a, nan=12345.0), torch.nan_to_num(b, nan=12345.0))
    keep = np.ones(64, bool)
    keep[[5, 40]] = False
    _check(arr, theta[keep].astype(np.float64), ref[0].cpu().numpy()[keep], ref[1].cpu().numpy()[keep], ref[2].cpu().numpy()[keep])
    p.close()


def test_host_path_with_page_locked_outputs():
    """Page-locked output arrays: the kernel writes lp and corr_coef straight into host memory (no copy); same numbers as
    with ordinary numpy arrays."""
    import torch
    from bpl_next_b200 import Problem

    arr = H.small_problem("extended", seed=3, weighted=True, K=3)
    p = Problem(arr)
    C = 77
    theta = H.random_theta(p.D, C, seed=4, radius=1.0, dtype=np.float32)
    lp0, g0, c0 = p.logdensity_host(theta)
    th = torch.from_numpy(theta).pin_memory()
    lp = torch.full((C,), -7.0).pin_memory()
    gr = torch.zeros((C, p.D)).pin_memory()
    cc = torch.full((C,), -7.0).pin_memory()
    for _ in range(3):
        p.logdensity_host(th.numpy(), lp=lp.numpy(), grad=gr.numpy(), corr_coef=cc.numpy())
    assert np.array_equal(lp.numpy(), lp0) and np.array_equal(gr.numpy(), g0) and np.array_equal(cc.numpy(), c0)
    _check(arr, theta.astype(np.float64), lp.numpy().copy(), gr.numpy().copy(), cc.numpy().copy())
    p.close()


@pytest.mark.parametrize("model,kw", [("dixon_coles", dict()), ("extended", dict(weighted=True)),
                                      ("neutral", dict()), ("neutral_wc", dict(multi_conf=True, T=13, M=400))])
@pytest.mark.parametrize("chain_minor", [False, True])
def test_likelihood_only_entry_point(model, kw, chain_minor):
    """bplx_loglik_fwdbwd (the numpyro.factor route, SURVEY 8(b)): constrained per-team tables in; Poisson + tau terms,
    corr_coef and d loglik / d tables out -- against the oracle's restatement of the reference's rate / likelihood lines."""
    import torch
    from bpl_next_b200 import Problem

    arr = H.small_problem(model, seed=6, **kw)
    d = H.to_oracle(arr)
    p = Problem(arr)
    lay = p.loglik_layout
    Dl = sum(c for _, c, _ in lay.values())
    C = 45
    rng = np.random.default_rng(12)
    tabs = rng.normal(0, 0.5, (C, Dl))
    o, c, _ = lay["corr_coef_raw"]
    tabs[:, o] = rng.uniform(0.05, 0.95, C)
    t32 = torch.from_numpy(tabs.astype(np.float32)).cuda()
    if chain_minor:
        t32 = t32.t().contiguous()
    ll, grad, cc = p.loglik(t32, chain_minor=chain_minor)
    torch.cuda.synchronize()
    g = (grad.t() if chain_minor else grad).cpu().numpy()
    # oracle: autograd through the restated likelihood
    x = torch.tensor(tabs.astype(np.float32).astype(np.float64), requires_grad=True)
    scalar_sites = ("corr_coef_raw",) + (("home_advantage",) if model == "dixon_coles" else ())
    tab = {name: (x[:, off] if name in scalar_sites else x[:, off:off + cnt]) for name, (off, cnt, _) in lay.items()}
    ll_o, cc_o = om.likelihood_from_tables(d, tab)
    (g_o,) = torch.autograd.grad(ll_o.sum(), x)
    np.testing.assert_allclose(ll.cpu().numpy(), ll_o.detach().numpy(), rtol=LP_RTOL)
    np.testing.assert_allclose(cc.cpu().numpy(), cc_o.detach().numpy(), rtol=1e-4, atol=1e-6)
    err = np.abs(g - g_o.numpy()) / np.abs(g_o.numpy()).max(axis=1, keepdims=True)
    assert err.max() < GRAD_RTOL, err.max()
