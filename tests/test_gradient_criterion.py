"""CPU: the per-component error criterion of tests/helpers.py (|g_i - g_o,i| <= c 2^-24 kappa_i, the same for lp).

* ``models.gradient_scale`` is exact: the same pieces summed with their signs give the oracle's lp and gradient; on
  small problems lp_scale is the sum of |term| and kappa bounds the sum of |column| of the dense Jacobian of every
  elementary term (kappa counts each path a term takes to theta_i on its own).
* Calibration: both float32 restatements of the oracle pass it on every case (helpers.CRIT_C records their worst ratio).
* It is strict: each mutation of the float64 gradient below is rejected.
"""
import numpy as np
import pytest
import torch

from oracle import closed_form, datasets, models as om
from tests import helpers as H

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
    ("extended", dict(T=20, M=300, K=16)),
    ("neutral", dict(T=20, M=300, K=16)),
    ("neutral_wc", dict(T=20, M=300, K=5)),
    ("dynamic", dict(T=20, M=300, K=16, Cf=4)),
]
CONFIGS = [("config_2", "extended", 0.01, (0.3, 2.0)), ("config_3", "neutral_wc", 0.1, (0.3, 2.0)),
           ("config_4", "dynamic", None, (0.3, 0.8))]  # a 30-step walk of U(-2, 2) steps overflows float32 rates


def _case(model, kw, seed=3):
    kw = dict(kw)
    as_written = kw.pop("as_written", False)
    arr = H.small_problem(model, seed=seed, **kw)
    arr.as_written = as_written
    return H.to_oracle(arr)


def _D(d):
    return om.num_params(d.model, d.num_teams, d.num_covariates, d.num_conferences if d.model == "neutral_wc" else 0,
                         d.num_gameweeks)


def _config(name, model, eps):
    return H.to_oracle(H.from_training_data(model, getattr(datasets, name)(), epsilon=eps))


def _float32_restatements(d, theta):
    out = [("models float32", om.log_density_and_grad(d, theta, dtype=torch.float32))]
    if d.model != "dynamic":
        out.append(("closed_form float32", closed_form.ClosedForm(d, torch.float32)(theta)))
    return out


# ---- gradient_scale is exact ------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,kw", CASES[:11])
def test_terms_sum_to_the_oracle(model, kw):
    d = _case(model, kw)
    theta = H.random_theta(_D(d), 4, seed=11, radius=2.0)
    lp_o, g_o, _ = om.log_density_and_grad(d, theta)
    kappa, lp_scale, g, lp = om._gradient_terms(d, theta)
    np.testing.assert_allclose(lp, lp_o, rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(g, g_o, rtol=0, atol=1e-12 * np.abs(g_o).max())
    assert (np.abs(g_o) <= kappa * (1 + 1e-12) + 1e-12).all() and (np.abs(lp_o) <= lp_scale * (1 + 1e-12)).all()


def _all_terms(d, th):
    """Every elementary term of the log density as one vector (the definition gradient_scale follows)."""
    pri = om._prior_terms(d, th)
    _, det = om.log_density(d, th)
    lh, la = det["lam_h"], det["lam_a"]
    w = torch.ones(d.num_matches, dtype=th.dtype) if d.weights is None else torch.as_tensor(d.weights, dtype=th.dtype)
    yh = torch.as_tensor(d.home_goals, dtype=th.dtype)
    ya = torch.as_tensor(d.away_goals, dtype=th.dtype)
    tau = om.dixon_coles_correlation_term(d.home_goals, d.away_goals, lh, la, det["corr_coef"], w)
    const = -w * (torch.lgamma(yh + 1) + torch.lgamma(ya + 1))
    return torch.cat([pri, w * yh * torch.log(lh), -w * lh, w * ya * torch.log(la), -w * la,
                      const.expand_as(lh), tau], dim=-1)


@pytest.mark.parametrize("model,kw", CASES[:11] + [("neutral_wc", dict(T=6, M=50, K=16, multi_conf=True))])
def test_kappa_bounds_the_dense_jacobian(model, kw):
    d = _case(model, kw)
    theta = H.random_theta(_D(d), 2, seed=7, radius=1.5)
    kappa, lp_scale = om.gradient_scale(d, theta)
    for c in range(2):
        th = torch.tensor(theta[c:c + 1])
        J = torch.autograd.functional.jacobian(lambda t: _all_terms(d, t)[0], th)[:, 0, :]
        assert (J.abs().sum(0).numpy() <= kappa[c] * (1 + 1e-12) + 1e-12).all()
        np.testing.assert_allclose(lp_scale[c], _all_terms(d, th).abs().sum().item(), rtol=1e-12)


# ---- calibration: the float32 restatements pass ---------------------------------------------------------------------
@pytest.mark.parametrize("model,kw", CASES)
@pytest.mark.parametrize("radius", [0.5, 2.0])
def test_float32_restatements_pass(model, kw, radius):
    d = _case(model, kw)
    if model == "dynamic" and (d.num_gameweeks > 8 or d.num_covariates > 8) and radius > 1.0:
        pytest.skip("a 33-step walk or 16 covariates of U(-2,2) overflow float32 rates")
    theta = H.random_theta(_D(d), 16, seed=11, radius=radius, dtype=np.float32).astype(np.float64)
    for name, (lp, g, _) in _float32_restatements(d, theta):
        H.assert_criterion(d, theta, lp, g, name)


@pytest.mark.parametrize("seed", range(0, 40, 3))
def test_float32_restatements_pass_random_problems(seed):
    """The randomised problems test_logdensity_gpu.py runs on the GPU (33 chains, radius 0.8)."""
    from tests.test_plan_random import _random_problem

    model, kw = _random_problem(seed)
    d = H.to_oracle(H.small_problem(model, seed=100 + seed, **kw))
    theta = H.random_theta(_D(d), 33, seed=seed, radius=0.8, dtype=np.float32).astype(np.float64)
    for name, (lp, g, _) in _float32_restatements(d, theta):
        H.assert_criterion(d, theta, lp, g, name)


@pytest.mark.parametrize("name,model,eps,radii", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_float32_restatements_pass_configs(name, model, eps, radii):
    d = _config(name, model, eps)
    for radius in radii:
        theta = H.random_theta(_D(d), 4, seed=21, radius=radius, dtype=np.float32).astype(np.float64)
        for what, (lp, g, _) in _float32_restatements(d, theta):
            H.assert_criterion(d, theta, lp, g, f"{what} radius {radius}")


# ---- the criterion rejects small errors -----------------------------------------------------------------------------
def _rejects(d, theta, lp, g):
    return len(H.criterion_failures(d, theta, lp, g)) > 0


def _site(d, name):
    lay = om.layout_offsets(om.site_layout(d.model, d.num_teams, d.num_covariates,
                                           d.num_conferences if d.model == "neutral_wc" else 0, d.num_gameweeks))
    o, shape, _ = lay[name]
    return o, shape


MUTATION_CASES = [("extended", dict(weighted=True, K=3)), ("neutral", dict(K=2)),
                  ("neutral_wc", dict(multi_conf=True, K=2, T=13, M=400)), ("dynamic", dict(Cf=4, T=5, M=90))]


@pytest.mark.parametrize("model,kw", MUTATION_CASES)
@pytest.mark.parametrize("radius", [0.5, 2.0])
def test_mutations_are_rejected(model, kw, radius):
    d = _case(model, kw)
    theta = H.random_theta(_D(d), 8, seed=11, radius=radius)
    lp_o, g_o, _ = om.log_density_and_grad(d, theta)
    assert not _rejects(d, theta, lp_o, g_o)
    o_a, shape_a = _site(d, "standardised_attack")
    team = 1 if model != "dynamic" else (d.num_gameweeks - 2) * d.num_teams + 1
    g = g_o.copy()
    g[:, o_a + team] *= 1.0 + 1e-3
    assert _rejects(d, theta, lp_o, g), "one team's standardised_attack x (1 + 1e-3)"
    o_r, _ = _site(d, "corr_coef_raw")
    g = g_o.copy()
    g[:, o_r] *= 1.01
    assert _rejects(d, theta, lp_o, g), "corr_coef_raw x 1.01"
    g = g_o.copy()
    g[:, [o_a + team, o_a + team + 1]] = g[:, [o_a + team + 1, o_a + team]]
    assert _rejects(d, theta, lp_o, g), "two teams' standardised_attack entries swapped"
    if model == "dynamic":  # every entry of the last gameweek x 1.01
        G, T = d.num_gameweeks, d.num_teams
        g = g_o.copy()
        for name, shape, _ in om.site_layout("dynamic", T, d.num_covariates, 0, G):
            if shape and shape[0] == G:
                o, _ = _site(d, name)
                n = int(np.prod(shape[1:])) if len(shape) > 1 else 1
                g[:, o + (G - 1) * n:o + G * n] *= 1.01
        assert _rejects(d, theta, lp_o, g), "last gameweek x 1.01"


@pytest.mark.parametrize("model,kw", MUTATION_CASES + [("dixon_coles", dict())])
def test_dropped_bound_fixup_is_rejected(model, kw, monkeypatch):
    """corr_coef = LB + r (UB - LB) with LB, UB the extreme rates' bounds: a gradient that treats the bounds as constants
    (no arg-max fix-up) must fail."""
    d = _case(model, kw)
    theta = H.random_theta(_D(d), 8, seed=11, radius=1.0)
    lp_o, _, _ = om.log_density_and_grad(d, theta)
    bounds = om.compute_corr_coef_bounds
    monkeypatch.setattr(om, "compute_corr_coef_bounds", lambda lh, la: tuple(b.detach() for b in bounds(lh, la)))
    _, g_nofix, _ = om.log_density_and_grad(d, theta)
    monkeypatch.undo()
    assert _rejects(d, theta, lp_o, g_nofix)


@pytest.mark.parametrize("model", ["extended", "neutral", "neutral_wc", "dynamic"])
def test_covariate_coefficient_mutation_is_rejected(model):
    kw = dict(T=20, M=300, K=16) if model != "dynamic" else dict(T=20, M=300, K=16, Cf=4)
    d = _case(model, kw)
    theta = H.random_theta(_D(d), 8, seed=11, radius=0.5)
    lp_o, g_o, _ = om.log_density_and_grad(d, theta)
    o, _ = _site(d, "attack_coefficients")
    for k in (0, 15):
        g = g_o.copy()
        g[:, o + k] *= 1.01
        assert _rejects(d, theta, lp_o, g), f"attack_coefficients[{k}] x 1.01"
