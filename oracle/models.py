"""Restatement of the five bpl-next ``_model`` log-densities in unconstrained space.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``: pinned to the reference's source run under stand-ins for jax /
numpyro, ``oracle/ref_shim.py``; numpyro's own arithmetic is restated, not pinned).

Written with torch so that the same lines give (a) float64 values + autograd gradients for parity
(``jax.grad`` of numpyro's ``potential_energy`` is what the reference runs) and (b) a float32,
multi-threaded CPU baseline.  Everything is batched over a leading chain axis: ``theta [C, D]``.

numpyro conventions restated here (numpyro 0.13.2, not vendored in /root/reference):
  * ``potential_energy = -(sum site log_prob + sum log|det J|)`` on unconstrained values;
    ``biject_to(positive) = exp``; ``biject_to(unit_interval / interval(0,1)) = clipped sigmoid``.
  * ``LocScaleReparam(centered=0)``: latent ``<x>_decentered ~ N(0,1)``; ``x = loc + scale*dec``.
  * ``plate`` + ``handlers.scale(scale=w)`` -> ``w * log_prob`` elementwise, then summed.
  * ``Poisson.log_prob(k) = log(rate)*k - lgamma(k+1) - rate``.

The flat layout of ``theta`` is model-declaration order with the scalar hyper-parameters first;
``site_layout`` returns it so tests can compare it with the layout the C library reports.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
LOG2 = math.log(2.0)

MODELS = ("dixon_coles", "extended", "neutral", "neutral_wc", "dynamic")


# --------------------------------------------------------------------------------------
# data container
# --------------------------------------------------------------------------------------
@dataclass
class MatchData:
    """Model arguments after the host-side prep each ``fit`` does (index arrays, weights).

    Mirrors the positional arguments of the reference ``_model`` functions
    (``dixon_coles.py:39-45``, ``extended_dixon_coles.py:78-88``, ``neutral_dixon_coles.py:102-114``,
    ``neutral_dixon_coles_WC.py:83-98``, ``dynamic_dixon_coles.py:63-73``).
    """

    model: str
    num_teams: int
    home_team: np.ndarray
    away_team: np.ndarray
    home_goals: np.ndarray
    away_goals: np.ndarray
    weights: Optional[np.ndarray] = None  # None -> unweighted (``to_event(1)`` branch)
    neutral_venue: Optional[np.ndarray] = None
    home_conf: Optional[np.ndarray] = None
    away_conf: Optional[np.ndarray] = None
    num_conferences: int = 0
    covariates: Optional[np.ndarray] = None  # raw [T, K]; standardised inside like the reference
    covariates_prestandardised: bool = False  # True: `covariates` already went through :124-127
    gameweek: Optional[np.ndarray] = None
    num_gameweeks: int = 0
    walk: str = "intended"  # dynamic only: "intended" | "as_written" (SURVEY Appendix D1)

    @property
    def num_covariates(self) -> int:
        return 0 if self.covariates is None else int(np.asarray(self.covariates).shape[1])

    @property
    def num_matches(self) -> int:
        return int(len(self.home_team))


# --------------------------------------------------------------------------------------
# weights (host side of each fit / _model)
# --------------------------------------------------------------------------------------
def weights_extended(time_diff, epsilon, rescale_weights=False, num_matches=None):
    """``extended_dixon_coles.py:202-205``; ``None`` when ``epsilon is None`` (``:216-217``)."""
    if epsilon is None:
        return None
    w = np.exp(-float(epsilon) * np.asarray(time_diff, dtype=np.float64))
    if rescale_weights:
        w = w.shape[0] * w / w.sum()
    return w


def weights_neutral(num_matches, time_diff, epsilon, game_weights, rescale_weights=False):
    """``neutral_dixon_coles.py:251-257``."""
    w = np.ones(num_matches, dtype=np.float64)
    if epsilon is not None:
        w = w * np.exp(-float(epsilon) * np.asarray(time_diff, dtype=np.float64))
        if rescale_weights:
            w = num_matches * w / w.sum()
    return w * np.asarray(game_weights, dtype=np.float64)


def weights_wc(num_matches, time_diff, epsilon, game_weights, rescale_weights=False):
    """``neutral_dixon_coles_WC.py:205-207`` (rescale applied after game_weights here)."""
    w = np.exp(-float(epsilon) * np.asarray(time_diff, dtype=np.float64)) * np.asarray(
        game_weights, dtype=np.float64
    )
    if rescale_weights:
        w = num_matches * w / w.sum()
    return w


def standardise_covariates(X):
    """``extended_dixon_coles.py:124-127`` (population std, axis 0)."""
    X = np.asarray(X, dtype=np.float64)
    return (X - X.mean(axis=0)) / X.std(axis=0)


# --------------------------------------------------------------------------------------
# theta layout
# --------------------------------------------------------------------------------------
def site_layout(model: str, T: int, K: int = 0, Cf: int = 0, G: int = 0) -> List[Tuple[str, Tuple[int, ...], str]]:
    """Ordered (site name, shape, transform) of the flat unconstrained vector.

    transform in {"real", "exp", "sigmoid"}.  Site names are numpyro's latent names
    (``*_decentered`` for LocScaleReparam'd sites).
    """
    r, e, s = "real", "exp", "sigmoid"
    if model == "dixon_coles":  # dixon_coles.py:46-78
        return [
            ("home_advantage", (), r), ("mean_defence", (), r),
            ("std_attack", (), e), ("std_defence", (), e),
            ("attack_decentered", (T,), r), ("defence_decentered", (T,), r),
            ("corr_coef_raw", (), s),
        ]
    if model == "extended":  # extended_dixon_coles.py:112-235
        return [
            ("mean_home_advantage", (), r), ("std_home_advantage", (), e), ("mean_defence", (), r),
            ("std_attack", (), e), ("std_defence", (), e),
            ("attack_coefficients", (K,), r), ("defence_coefficients", (K,), r),
            ("u", (), s),
            ("standardised_attack", (T,), r), ("standardised_defence", (T,), r),
            ("home_advantage_decentered", (T,), r),
            ("corr_coef_raw", (), s),
        ]
    if model in ("neutral", "neutral_wc"):  # neutral_dixon_coles.py:136-272 / ..._WC.py:99-219
        lay = [
            ("mean_defence", (), r), ("std_attack", (), e), ("std_defence", (), e),
            ("mean_home_attack", (), r), ("mean_away_attack", (), r),
            ("mean_home_defence", (), r), ("mean_away_defence", (), r),
            ("std_home_attack", (), e), ("std_away_attack", (), e),
            ("std_home_defence", (), e), ("std_away_defence", (), e),
            ("u", (), s),
            ("attack_coefficients", (K,), r), ("defence_coefficients", (K,), r),
            ("standardised_attack", (T,), r), ("standardised_defence", (T,), r),
            ("home_attack_decentered", (T,), r), ("away_attack_decentered", (T,), r),
            ("home_defence_decentered", (T,), r), ("away_defence_decentered", (T,), r),
        ]
        if model == "neutral_wc":
            lay.append(("confederation_strength_decentered", (Cf,), r))
        lay.append(("corr_coef_raw", (), s))
        return lay
    if model == "dynamic":  # dynamic_dixon_coles.py:74-241
        return [
            ("mean_home_attack", (G,), r), ("mean_away_attack", (G,), r),
            ("mean_home_defence", (G,), r), ("mean_away_defence", (G,), r),
            ("std_home_attack", (G,), e), ("std_away_attack", (G,), e),
            ("std_home_defence", (G,), e), ("std_away_defence", (G,), e),
            ("std_attack", (G,), e), ("std_defence", (G,), e),
            ("mean_defence", (), r),
            ("attack_coefficients", (K,), r), ("defence_coefficients", (K,), r),
            ("u", (G, T), s),
            ("standardised_attack", (G, T), r), ("standardised_defence", (G, T), r),
            ("home_attack_decentered", (G, T), r), ("away_attack_decentered", (G, T), r),
            ("home_defence_decentered", (G, T), r), ("away_defence_decentered", (G, T), r),
            ("corr_coef_raw", (), s),
        ]
    raise ValueError(f"unknown model {model!r}")


def layout_offsets(layout) -> Dict[str, Tuple[int, Tuple[int, ...], str]]:
    out, off = {}, 0
    for name, shape, tr in layout:
        n = int(np.prod(shape)) if shape else 1
        out[name] = (off, shape, tr)
        off += n
    out["__D__"] = (off, (), "")
    return out


def num_params(model, T, K=0, Cf=0, G=0) -> int:
    return layout_offsets(site_layout(model, T, K, Cf, G))["__D__"][0]


# --------------------------------------------------------------------------------------
# numpyro distribution / transform arithmetic
# --------------------------------------------------------------------------------------
def _normal_lp(x, loc, scale):
    """numpyro ``Normal.log_prob``: -0.5*((x-loc)/scale)^2 - log(sqrt(2 pi) * scale)."""
    if not torch.is_tensor(scale):
        scale = torch.as_tensor(scale, dtype=x.dtype)
    z = (x - loc) / scale
    return -0.5 * z * z - torch.log(scale) - LOG_SQRT_2PI


def _halfnormal_lp(x, scale):
    """numpyro ``HalfNormal.log_prob`` = Normal(0, scale).log_prob + log 2."""
    return _normal_lp(x, 0.0, scale) + LOG2


def _beta_lp(x, c1, c0):
    """numpyro ``Beta.log_prob`` via the 2-component Dirichlet (xlogy form)."""
    lognorm = math.lgamma(c1) + math.lgamma(c0) - math.lgamma(c1 + c0)
    return torch.xlogy(torch.as_tensor(c1 - 1.0, dtype=x.dtype), x) + torch.xlogy(
        torch.as_tensor(c0 - 1.0, dtype=x.dtype), 1.0 - x
    ) - lognorm


def _poisson_lp(k, rate):
    """numpyro ``Poisson.log_prob``."""
    return torch.log(rate) * k - torch.lgamma(k + 1.0) - rate


def _exp_site(x):
    """ExpTransform: value, log|det J| = x."""
    return torch.exp(x), x


def _sigmoid_site(x):
    """SigmoidTransform: clipped expit, log|det J| = -softplus(x) - softplus(-x)."""
    fi = torch.finfo(x.dtype)
    val = torch.clamp(torch.sigmoid(x), min=fi.tiny, max=1.0 - fi.eps)
    sp = torch.nn.functional.softplus
    return val, -sp(x) - sp(-x)


# --------------------------------------------------------------------------------------
# bpl/_util.py
# --------------------------------------------------------------------------------------
def compute_corr_coef_bounds(lam_h, lam_a):
    """``bpl/_util.py:17-31``: UB = min(min 1/(lh*la), 1); LB = max(max -1/lh, max -1/la)."""
    one = torch.ones_like(lam_h[..., 0])
    UB = torch.minimum((1.0 / (lam_h * lam_a)).amin(dim=-1), one)
    LB = torch.maximum((-1.0 / lam_h).amax(dim=-1), (-1.0 / lam_a).amax(dim=-1))
    return LB, UB


def dixon_coles_correlation_term(home_goals, away_goals, lam_h, lam_a, corr_coef, weights=None, tol=0.0):
    """``bpl/_util.py:35-93``: w * log(clip(tau, tol)) on the four low-score cells, 0 elsewhere."""
    hg = np.asarray(home_goals)
    ag = np.asarray(away_goals)
    if weights is None:
        weights = torch.ones(len(hg), dtype=lam_h.dtype)
    corr = torch.zeros_like(lam_h)
    c = corr_coef[..., None]

    def put(mask, tau):
        nonlocal corr
        idx = torch.as_tensor(np.nonzero(mask)[0], dtype=torch.long)
        if idx.numel() == 0:
            return
        val = weights[idx] * torch.log(torch.clamp(tau(idx), min=tol))
        corr = corr.index_copy(-1, idx, val.expand(corr.shape[:-1] + (idx.numel(),)))

    put((hg == 0) & (ag == 0), lambda i: 1.0 - c * lam_h[..., i] * lam_a[..., i])
    put((hg == 1) & (ag == 0), lambda i: 1.0 + c * lam_a[..., i])
    put((hg == 0) & (ag == 1), lambda i: 1.0 + c * lam_h[..., i])
    put((hg == 1) & (ag == 1), lambda i: (1.0 - c).expand(c.shape[:-1] + (i.numel(),)))
    return corr


# --------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------
def _split(theta, layout):
    off = layout_offsets(layout)
    out = {}
    for name, (o, shape, tr) in off.items():
        if name == "__D__":
            continue
        n = int(np.prod(shape)) if shape else 1
        x = theta[..., o : o + n]
        out[name] = x[..., 0] if shape == () else x.reshape(theta.shape[:-1] + tuple(shape))
    return out


def _likelihood(d: MatchData, lam_h, lam_a, corr_raw, dtype):
    """Poisson terms (+ optional weights) and the tau factor; returns (loglik [C], corr_coef [C])."""
    hg = torch.as_tensor(np.asarray(d.home_goals), dtype=dtype)
    ag = torch.as_tensor(np.asarray(d.away_goals), dtype=dtype)
    w = None if d.weights is None else torch.as_tensor(np.asarray(d.weights), dtype=dtype)
    lp_h = _poisson_lp(hg, lam_h)
    lp_a = _poisson_lp(ag, lam_a)
    if w is not None:  # plate("data") + handlers.scale(scale=weights)
        lp_h = lp_h * w
        lp_a = lp_a * w
    ll = lp_h.sum(-1) + lp_a.sum(-1)
    LB, UB = compute_corr_coef_bounds(lam_h, lam_a)
    corr_coef = LB + corr_raw * (UB - LB)
    corr = dixon_coles_correlation_term(d.home_goals, d.away_goals, lam_h, lam_a, corr_coef, w)
    return ll + corr.sum(-1), corr_coef


def _idx(a):
    return torch.as_tensor(np.asarray(a, dtype=np.int64))


_tap: Optional[list] = None  # while set (``_prior_terms``), every prior and Jacobian term a model adds is appended


def _term(x, parts=None):
    """One group of elementary prior / Jacobian terms (one per element of ``x``), as the model adds it to lp; ``parts``
    (summing to ``x``) are recorded in its place when ``x`` cancels inside itself."""
    if _tap is not None:
        _tap.extend([x] if parts is None else parts)
    return x


def _conditional_normal(zd, loc, s2):
    """N(zd | loc, sqrt(s2)) log-prob; recorded as the parts of its expanded square, so that the error scale sees
    zd and loc rather than their (possibly cancelling) difference."""
    x = _normal_lp(zd, loc, torch.sqrt(s2))
    parts = [-0.5 * zd * zd / s2, zd * loc / s2, -0.5 * loc * loc / s2, -0.5 * torch.log(s2) - LOG_SQRT_2PI]
    return _term(x, [p.expand_as(x) for p in parts])


def _prior_means(d: MatchData, mean_defence, beta_a, beta_d, dtype):
    """Attack/defence prior means, with covariates ``extended_dixon_coles.py:123-146``."""
    if d.covariates is not None:
        Xs = d.covariates if d.covariates_prestandardised else standardise_covariates(d.covariates)
        Xs = torch.as_tensor(np.asarray(Xs, dtype=np.float64), dtype=dtype)
        a_mean = torch.matmul(Xs, beta_a[..., None]).squeeze(-1)
        d_mean = mean_defence[..., None] + torch.matmul(Xs, beta_d[..., None]).squeeze(-1)
    else:
        a_mean = torch.zeros_like(mean_defence)[..., None]
        d_mean = mean_defence[..., None]
    return a_mean, d_mean


# --------------------------------------------------------------------------------------
# the five models.  Each returns (log_density [C], deterministics dict)
# --------------------------------------------------------------------------------------
def _dixon_coles(d: MatchData, theta):
    """``bpl/dixon_coles.py:39-84``."""
    T = d.num_teams
    s = _split(theta, site_layout("dixon_coles", T))
    dt = theta.dtype
    lp = _term(_normal_lp(s["home_advantage"], 0.1, 0.2)) + _term(_normal_lp(s["mean_defence"], 0.0, 1.0))
    std_a, j = _exp_site(s["std_attack"]); lp = lp + _term(_halfnormal_lp(std_a, 1.0)) + _term(j)
    std_d, j = _exp_site(s["std_defence"]); lp = lp + _term(_halfnormal_lp(std_d, 1.0)) + _term(j)
    lp = lp + _term(_normal_lp(s["attack_decentered"], 0.0, 1.0)).sum(-1)
    lp = lp + _term(_normal_lp(s["defence_decentered"], 0.0, 1.0)).sum(-1)
    attack = 0.0 + std_a[..., None] * s["attack_decentered"]
    defence = s["mean_defence"][..., None] + std_d[..., None] * s["defence_decentered"]
    h, a = _idx(d.home_team), _idx(d.away_team)
    lam_h = torch.exp(attack[..., h] - defence[..., a] + s["home_advantage"][..., None])
    lam_a = torch.exp(attack[..., a] - defence[..., h])
    raw, j = _sigmoid_site(s["corr_coef_raw"]); lp = lp + _term(_beta_lp(raw, 2.0, 2.0)) + _term(j)
    ll, cc = _likelihood(d, lam_h, lam_a, raw, dt)
    return lp + ll, {"attack": attack, "defence": defence, "home_advantage": s["home_advantage"],
                     "corr_coef": cc, "lam_h": lam_h, "lam_a": lam_a}


def _rho_block(s, lp):
    """u ~ Beta(2,4), rho = 2u-1, za ~ N(0,1), zd ~ N(rho za, sqrt(1-rho^2))
    (``extended_dixon_coles.py:152-174``)."""
    u, j = _sigmoid_site(s["u"]); lp = lp + _term(_beta_lp(u, 2.0, 4.0)) + _term(j)
    rho = 2.0 * u - 1.0
    za, zd = s["standardised_attack"], s["standardised_defence"]
    lp = lp + _term(_normal_lp(za, 0.0, 1.0)).sum(-1)
    lp = lp + _conditional_normal(zd, rho[..., None] * za, (1.0 - rho**2.0)[..., None]).sum(-1)
    return lp, rho


def _extended(d: MatchData, theta):
    """``bpl/extended_dixon_coles.py:78-248``."""
    T, K = d.num_teams, d.num_covariates
    s = _split(theta, site_layout("extended", T, K))
    dt = theta.dtype
    lp = _term(_normal_lp(s["mean_home_advantage"], 0.1, 0.2))
    std_ha, j = _exp_site(s["std_home_advantage"]); lp = lp + _term(_halfnormal_lp(std_ha, 1.0)) + _term(j)
    lp = lp + _term(_normal_lp(s["mean_defence"], 0.0, 1.0))
    std_a, j = _exp_site(s["std_attack"]); lp = lp + _term(_halfnormal_lp(std_a, 1.0)) + _term(j)
    std_d, j = _exp_site(s["std_defence"]); lp = lp + _term(_halfnormal_lp(std_d, 1.0)) + _term(j)
    if K:
        lp = lp + _term(_normal_lp(s["attack_coefficients"], 0.0, 1.0)).sum(-1)
        lp = lp + _term(_normal_lp(s["defence_coefficients"], 0.0, 1.0)).sum(-1)
    a_mean, d_mean = _prior_means(d, s["mean_defence"], s["attack_coefficients"], s["defence_coefficients"], dt)
    lp, rho = _rho_block(s, lp)
    lp = lp + _term(_normal_lp(s["home_advantage_decentered"], 0.0, 1.0)).sum(-1)
    home_adv = s["mean_home_advantage"][..., None] + std_ha[..., None] * s["home_advantage_decentered"]
    attack = a_mean + s["standardised_attack"] * std_a[..., None]
    defence = d_mean + s["standardised_defence"] * std_d[..., None]
    h, a = _idx(d.home_team), _idx(d.away_team)
    lam_h = torch.exp(attack[..., h] - defence[..., a] + home_adv[..., h])
    lam_a = torch.exp(attack[..., a] - defence[..., h])
    lam_h = torch.clamp(lam_h, max=15.0)  # :197-198
    lam_a = torch.clamp(lam_a, max=15.0)
    raw, j = _sigmoid_site(s["corr_coef_raw"]); lp = lp + _term(_beta_lp(raw, 2.0, 2.0)) + _term(j)
    ll, cc = _likelihood(d, lam_h, lam_a, raw, dt)
    return lp + ll, {"attack": attack, "defence": defence, "home_advantage": home_adv, "rho": rho,
                     "corr_coef": cc, "lam_h": lam_h, "lam_a": lam_a}


def _neutral_family(d: MatchData, theta, wc: bool):
    """``bpl/neutral_dixon_coles.py:102-283`` and ``bpl/neutral_dixon_coles_WC.py:83-232``."""
    T, K, Cf = d.num_teams, d.num_covariates, (d.num_conferences if wc else 0)
    s = _split(theta, site_layout("neutral_wc" if wc else "neutral", T, K, Cf))
    dt = theta.dtype
    lp = _term(_normal_lp(s["mean_defence"], 0.0, 1.0))
    std_a, j = _exp_site(s["std_attack"]); lp = lp + _term(_halfnormal_lp(std_a, 0.5)) + _term(j)
    std_d, j = _exp_site(s["std_defence"]); lp = lp + _term(_halfnormal_lp(std_d, 0.5)) + _term(j)
    lp = lp + _term(_normal_lp(s["mean_home_attack"], 0.1, 0.2)) + _term(_normal_lp(s["mean_away_attack"], -0.1, 0.2))
    lp = lp + _term(_normal_lp(s["mean_home_defence"], 0.1, 0.2)) + _term(_normal_lp(s["mean_away_defence"], -0.1, 0.2))
    stds = {}
    for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
        v, j = _exp_site(s["std_" + nm]); lp = lp + _term(_halfnormal_lp(v, 1.0)) + _term(j)
        stds[nm] = v
    if K:
        lp = lp + _term(_normal_lp(s["attack_coefficients"], 0.0, 1.0)).sum(-1)
        lp = lp + _term(_normal_lp(s["defence_coefficients"], 0.0, 1.0)).sum(-1)
    a_mean, d_mean = _prior_means(d, s["mean_defence"], s["attack_coefficients"], s["defence_coefficients"], dt)
    lp, rho = _rho_block(s, lp)
    eff = {}
    for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
        dec = s[nm + "_decentered"]
        lp = lp + _term(_normal_lp(dec, 0.0, 1.0)).sum(-1)
        eff[nm] = s["mean_" + nm][..., None] + stds[nm][..., None] * dec
    attack = a_mean + s["standardised_attack"] * std_a[..., None]
    defence = d_mean + s["standardised_defence"] * std_d[..., None]
    h, a = _idx(d.home_team), _idx(d.away_team)
    n = torch.as_tensor(1 - np.asarray(d.neutral_venue, dtype=np.int64), dtype=dt)
    eta_h = attack[..., h] - defence[..., a] + n * eff["home_attack"][..., h] - n * eff["away_defence"][..., a]
    eta_a = attack[..., a] - defence[..., h] + n * eff["away_attack"][..., a] - n * eff["home_defence"][..., h]
    det = {}
    if wc:  # confederation_strength ~ N(0,1), LocScaleReparam -> identity (..._WC.py:180-203)
        conf = s["confederation_strength_decentered"]
        lp = lp + _term(_normal_lp(conf, 0.0, 1.0)).sum(-1)
        hc, ac = _idx(d.home_conf), _idx(d.away_conf)
        eta_h = eta_h + conf[..., hc] - conf[..., ac]
        eta_a = eta_a + conf[..., ac] - conf[..., hc]
        det["confederation_strength"] = conf
    lam_h, lam_a = torch.exp(eta_h), torch.exp(eta_a)
    raw, j = _sigmoid_site(s["corr_coef_raw"]); lp = lp + _term(_beta_lp(raw, 2.0, 2.0)) + _term(j)
    ll, cc = _likelihood(d, lam_h, lam_a, raw, dt)
    det.update({"attack": attack, "defence": defence, "rho": rho, "corr_coef": cc, "lam_h": lam_h,
                "lam_a": lam_a, **eff})
    return lp + ll, det


def _dynamic(d: MatchData, theta):
    """``bpl/dynamic_dixon_coles.py:63-247``.

    ``walk="as_written"`` reproduces the reference exactly: ``attack``/``defence`` stay the zeros
    that ``jnp.empty`` returns because every ``.at[j].set`` result is discarded (``:192-218``), so
    the rates see only the venue effects.  ``walk="intended"`` is the cumulative random walk the
    code meant to build.
    """
    T, K, G = d.num_teams, d.num_covariates, d.num_gameweeks
    s = _split(theta, site_layout("dynamic", T, K, 0, G))
    dt = theta.dtype
    lp = _term(_normal_lp(s["mean_home_attack"], 0.1, 0.2)).sum(-1) + _term(_normal_lp(s["mean_away_attack"], -0.1, 0.2)).sum(-1)
    lp = lp + _term(_normal_lp(s["mean_home_defence"], 0.1, 0.2)).sum(-1) + _term(_normal_lp(s["mean_away_defence"], -0.1, 0.2)).sum(-1)
    stds = {}
    for nm in ("home_attack", "away_attack", "home_defence", "away_defence", "attack", "defence"):
        v, j = _exp_site(s["std_" + nm])
        lp = lp + (_term(_halfnormal_lp(v, 1.0)) + _term(j)).sum(-1)
        stds[nm] = v  # [C, G]
    lp = lp + _term(_normal_lp(s["mean_defence"], 0.0, 1.0))
    if K:
        lp = lp + _term(_normal_lp(s["attack_coefficients"], 0.0, 1.0)).sum(-1)
        lp = lp + _term(_normal_lp(s["defence_coefficients"], 0.0, 1.0)).sum(-1)
    a_mean, d_mean = _prior_means(d, s["mean_defence"], s["attack_coefficients"], s["defence_coefficients"], dt)
    u, j = _sigmoid_site(s["u"])  # [C, G, T]
    lp = lp + (_term(_beta_lp(u, 2.0, 4.0)) + _term(j)).sum((-1, -2))
    rho = 2.0 * u - 1.0
    za, zd = s["standardised_attack"], s["standardised_defence"]
    lp = lp + _term(_normal_lp(za, 0.0, 1.0)).sum((-1, -2))
    lp = lp + _conditional_normal(zd, rho * za, 1.0 - rho**2.0).sum((-1, -2))
    eff = {}
    for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
        dec = s[nm + "_decentered"]
        lp = lp + _term(_normal_lp(dec, 0.0, 1.0)).sum((-1, -2))
        eff[nm] = s["mean_" + nm][..., None] + stds[nm][..., None] * dec  # [C, G, T]
    step_a = za * stds["attack"][..., None]
    step_d = zd * stds["defence"][..., None]
    if d.walk == "intended":
        attack = torch.cumsum(step_a, dim=-2) + a_mean[..., None, :]
        defence = torch.cumsum(step_d, dim=-2) + d_mean[..., None, :]
    elif d.walk == "as_written":
        attack = torch.zeros_like(step_a)
        defence = torch.zeros_like(step_d)
    else:
        raise ValueError(d.walk)
    h, a, g = _idx(d.home_team), _idx(d.away_team), _idx(d.gameweek)
    n = torch.as_tensor(1 - np.asarray(d.neutral_venue, dtype=np.int64), dtype=dt)
    lam_h = torch.exp(attack[..., g, h] - defence[..., g, a]
                      + n * eff["home_attack"][..., g, h] - n * eff["away_defence"][..., g, a])
    lam_a = torch.exp(attack[..., g, a] - defence[..., g, h]
                      + n * eff["away_attack"][..., g, a] - n * eff["home_defence"][..., g, h])
    raw, j = _sigmoid_site(s["corr_coef_raw"])  # Uniform(0,1): log_prob 0 (:241)
    lp = lp + _term(j)
    ll, cc = _likelihood(d, lam_h, lam_a, raw, dt)
    return lp + ll, {"attack": attack, "defence": defence, "rho": rho, "corr_coef": cc,
                     "lam_h": lam_h, "lam_a": lam_a, **eff}


def log_density(d: MatchData, theta: torch.Tensor):
    """log joint density (= -potential_energy) of unconstrained ``theta [..., D]``."""
    if d.model == "dixon_coles":
        return _dixon_coles(d, theta)
    if d.model == "extended":
        return _extended(d, theta)
    if d.model == "neutral":
        return _neutral_family(d, theta, wc=False)
    if d.model == "neutral_wc":
        return _neutral_family(d, theta, wc=True)
    if d.model == "dynamic":
        return _dynamic(d, theta)
    raise ValueError(d.model)


def log_density_and_grad(d: MatchData, theta, dtype=torch.float64):
    """Returns (lp [C], grad [C, D], corr_coef [C]) as numpy arrays; gradient by autograd."""
    th = torch.as_tensor(np.asarray(theta), dtype=dtype).clone().requires_grad_(True)
    lp, det = log_density(d, th)
    (g,) = torch.autograd.grad(lp.sum(), th)
    return lp.detach().numpy(), g.numpy(), det["corr_coef"].detach().numpy()


# --------------------------------------------------------------------------------------
# error scale of a float32 evaluation: sum over the elementary terms of |d term / d theta_i|
# --------------------------------------------------------------------------------------
def _prior_terms(d: MatchData, theta):
    """Every prior and Jacobian term of the log density, ``[C, N]`` (the likelihood's terms are not in it)."""
    global _tap
    _tap = []
    try:
        log_density(d, theta)
        C = theta.shape[0]
        return torch.cat([x.reshape(C, -1) for x in _tap], dim=-1)
    finally:
        _tap = None


def _rate_jacobian(d: MatchData, theta):
    """d eta / d theta of the log-rates eta_h, eta_a of every match (before any clip), sparse: per side a list of
    (theta index [M], value [C, M]); row m of the Jacobian is the sum over the list (an index may repeat)."""
    model, T, K, G = d.model, d.num_teams, d.num_covariates, d.num_gameweeks
    Cf = d.num_conferences if model == "neutral_wc" else 0
    lay = site_layout(model, T, K, Cf, G)
    off = layout_offsets(lay)
    s = _split(theta, lay)
    C = theta.shape[0]
    h, a = np.asarray(d.home_team, np.int64), np.asarray(d.away_team, np.int64)
    M = len(h)
    o = lambda name: off[name][0]  # noqa: E731
    full = lambda i: np.full(M, i, np.int64)  # noqa: E731
    ones = torch.ones((C, M), dtype=theta.dtype)
    X = None
    if K:
        X = np.asarray(d.covariates if d.covariates_prestandardised else standardise_covariates(d.covariates), np.float64)
    n = ones if model in ("dixon_coles", "extended") else ones * torch.as_tensor(
        1 - np.asarray(d.neutral_venue, np.int64), dtype=theta.dtype)
    jh, ja = [], []
    if model == "dynamic":
        g = np.asarray(d.gameweek, np.int64)
        sa, sd = torch.exp(s["std_attack"]), torch.exp(s["std_defence"])  # [C, G]

        def strength(side, t, sign, out):  # sign * attack[g, t] or sign * defence[g, t]: the walk up to gameweek g
            if d.walk == "as_written":  # (attack and defence stay zero)
                return
            z, ls, sg = ("standardised_" + side, "std_" + side, sa if side == "attack" else sd)
            for j in range(G):
                on = torch.as_tensor((j <= g).astype(np.float64), dtype=theta.dtype)
                out.append((o(z) + j * T + t, sign * sg[:, j, None] * on))
                out.append((full(o(ls) + j), sign * sg[:, j, None] * s[z][:, j, t] * on))
            if side == "defence":
                out.append((full(o("mean_defence")), sign * ones))
            for k in range(K):
                out.append((full(o(side + "_coefficients") + k), sign * torch.as_tensor(X[t, k], dtype=theta.dtype).expand(C, M)))

        def effect(nm, t, coef, out):  # coef * effect[g, t]
            sg = torch.exp(s["std_" + nm])
            out.append((o("mean_" + nm) + g, coef))
            out.append((o("std_" + nm) + g, coef * sg[:, g] * s[nm + "_decentered"][:, g, t]))
            out.append((o(nm + "_decentered") + g * T + t, coef * sg[:, g]))

        strength("attack", h, 1.0, jh); strength("defence", a, -1.0, jh)
        effect("home_attack", h, n, jh); effect("away_defence", a, -n, jh)
        strength("attack", a, 1.0, ja); strength("defence", h, -1.0, ja)
        effect("away_attack", a, n, ja); effect("home_defence", h, -n, ja)
        return jh, ja
    dc = model == "dixon_coles"
    za_n, zd_n = ("attack_decentered", "defence_decentered") if dc else ("standardised_attack", "standardised_defence")
    sa, sd = torch.exp(s["std_attack"]), torch.exp(s["std_defence"])

    def attack(t, out):
        out.append((o(za_n) + t, sa[:, None] * ones))
        out.append((full(o("std_attack")), sa[:, None] * s[za_n][:, t]))
        for k in range(K):
            out.append((full(o("attack_coefficients") + k), torch.as_tensor(X[t, k], dtype=theta.dtype).expand(C, M)))

    def minus_defence(t, out):
        out.append((o(zd_n) + t, -sd[:, None] * ones))
        out.append((full(o("std_defence")), -sd[:, None] * s[zd_n][:, t]))
        out.append((full(o("mean_defence")), -ones))
        for k in range(K):
            out.append((full(o("defence_coefficients") + k), -torch.as_tensor(X[t, k], dtype=theta.dtype).expand(C, M)))

    def effect(nm, mean, std, t, coef, out):  # coef * (mean + std * decentred[t])
        sg = torch.exp(s[std])
        out.append((full(o(mean)), coef))
        out.append((full(o(std)), coef * sg[:, None] * s[nm + "_decentered"][:, t]))
        out.append((o(nm + "_decentered") + t, coef * sg[:, None]))

    attack(h, jh); minus_defence(a, jh); attack(a, ja); minus_defence(h, ja)
    if dc:
        jh.append((full(o("home_advantage")), ones))
    elif model == "extended":
        effect("home_advantage", "mean_home_advantage", "std_home_advantage", h, ones, jh)
    else:
        for nm, t, sign, out in (("home_attack", h, 1, jh), ("away_defence", a, -1, jh),
                                 ("away_attack", a, 1, ja), ("home_defence", h, -1, ja)):
            effect(nm, "mean_" + nm, "std_" + nm, t, sign * n, out)
    if Cf:
        hc, ac = np.asarray(d.home_conf, np.int64), np.asarray(d.away_conf, np.int64)
        oc = o("confederation_strength_decentered")
        jh += [(oc + hc, ones), (oc + ac, -ones)]
        ja += [(oc + ac, ones), (oc + hc, -ones)]
    return jh, ja


def _gradient_terms(d: MatchData, theta):
    """float64 (kappa [C, D], lp scale [C], gradient [C, D], lp [C]): kappa_i = sum over the elementary terms, and
    over the paths by which a term reaches theta_i, of |d term / d theta_i|; the lp scale = sum of |term|.  The
    gradient and lp are the same pieces summed with their signs (they equal ``log_density_and_grad``: a check of the
    decomposition).

    Elementary terms: per match w y_h log lam_h, -w lam_h, w y_a log lam_a, -w lam_a, -w log(y_h! y_a!) and, for low
    scores, w log tau (tau through corr_coef and its bounds); every prior and Jacobian term, one per element (the
    conditional normal of the standardised defence as the parts of its expanded square).  A match term reaches theta
    through eta_h, eta_a and corr_coef, and each rate through each table entry it reads (attack[h], confederation
    strength[home conf], ... -- separately even when two cancel, as two entries of one confederation do): float32
    evaluates each path on its own.  The match terms are differentiated through the sparse rows of d eta / d theta (per
    chain, ``scipy.sparse``), the prior terms site by site: inside one site every prior term reads at most one element,
    so a forward derivative along the whole site gives each term's derivative and a reverse pass weighted by its sign
    sums their moduli."""
    import scipy.sparse as sp

    th = torch.as_tensor(np.asarray(theta), dtype=torch.float64).clone().requires_grad_(True)
    C, D = th.shape
    lp_o, det = log_density(d, th)
    cc = det["corr_coef"]
    (dc_dth,) = torch.autograd.grad(cc.sum(), th)  # d corr_coef / d theta: raw and the two arg-max matches' rates
    dc_dth = dc_dth.numpy()
    lam_h, lam_a, c = det["lam_h"].detach(), det["lam_a"].detach(), cc.detach()[:, None]
    # ---- match terms: derivatives with respect to eta_h, eta_a and c (the rates are clipped only in "extended") ----
    M = d.num_matches
    w = torch.ones(M, dtype=torch.float64) if d.weights is None else torch.as_tensor(np.asarray(d.weights, np.float64))
    hg, ag = np.asarray(d.home_goals, np.int64), np.asarray(d.away_goals, np.int64)
    yh, ya = torch.as_tensor(hg, dtype=torch.float64), torch.as_tensor(ag, dtype=torch.float64)
    fh = (lam_h < 15.0).double() if d.model == "extended" else torch.ones_like(lam_h)
    fa = (lam_a < 15.0).double() if d.model == "extended" else torch.ones_like(lam_a)
    t_pois = [w * yh * torch.log(lam_h), -w * lam_h, w * ya * torch.log(lam_a), -w * lam_a,
              (-w * (torch.lgamma(yh + 1.0) + torch.lgamma(ya + 1.0))).expand(C, M)]
    k00 = torch.as_tensor((hg == 0) & (ag == 0)).double()
    k10 = torch.as_tensor((hg == 1) & (ag == 0)).double()
    k01 = torch.as_tensor((hg == 0) & (ag == 1)).double()
    k11 = torch.as_tensor((hg == 1) & (ag == 1)).double()
    low = (k00 + k10 + k01 + k11) > 0
    x = lam_h * lam_a
    tau = 1.0 + c * (-k00 * x + k10 * lam_a + k01 * lam_h - k11)  # 1 - c x, 1 + c lam_a, 1 + c lam_h, 1 - c
    tau = torch.where(low, tau, torch.ones_like(tau))
    t_tau = w * torch.log(tau) * low
    a_h = w * (yh - lam_h) * fh  # Poisson terms, d / d eta_h (both terms: |.| taken per term below)
    p_h = w * (yh + lam_h) * fh  # sum of the two terms' moduli
    a_a, p_a = w * (ya - lam_a) * fa, w * (ya + lam_a) * fa
    q_h = w * c * (-k00 * x + k01 * lam_h) / tau * fh  # tau term, d / d eta_h
    q_a = w * c * (-k00 * x + k10 * lam_a) / tau * fa
    q_c = w * (-k00 * x + k10 * lam_a + k01 * lam_h - k11) / tau  # d / d c
    # ---- prior terms --------------------------------------------------------------------------------------------
    pri = _prior_terms(d, th.detach())
    kappa = np.zeros((C, D))
    grad = np.zeros((C, D))
    f = lambda t: _prior_terms(d, t)  # noqa: E731
    _, vjp = torch.func.vjp(f, th.detach())
    grad += vjp(torch.ones_like(pri))[0].numpy()
    off = layout_offsets(site_layout(d.model, d.num_teams, d.num_covariates,
                                     d.num_conferences if d.model == "neutral_wc" else 0, d.num_gameweeks))
    for name, (o, shape, _) in off.items():
        n = int(np.prod(shape)) if shape else 1
        if name == "__D__" or n == 0:
            continue
        e = torch.zeros_like(th.detach())
        e[:, o:o + n] = 1.0
        _, along = torch.func.jvp(f, (th.detach(),), (e,))
        kappa[:, o:o + n] += vjp(torch.sign(along))[0][:, o:o + n].numpy()
    lp_scale = pri.abs().sum(-1).numpy() + sum(t.abs().sum(-1) for t in t_pois).numpy() + t_tau.abs().sum(-1).numpy()
    lp = pri.sum(-1).numpy() + sum(t.sum(-1) for t in t_pois).numpy() + t_tau.sum(-1).numpy()
    # ---- match terms through the sparse rate Jacobian, chain by chain ---------------------------------------------
    jh, ja = _rate_jacobian(d, th.detach())
    rows = np.arange(M)

    def csr(parts, c_, absolute=False):  # duplicate (row, column) pairs are summed: after |.| with absolute=True
        r = np.concatenate([rows] * len(parts))
        i = np.concatenate([np.broadcast_to(ix, (M,)) for ix, _ in parts])
        v = np.concatenate([val[c_].numpy() for _, val in parts])
        return sp.csr_matrix((np.abs(v) if absolute else v, (r, i)), shape=(M, D))

    lowi = np.nonzero(low.numpy())[0]
    for c_ in range(C):
        Jh, Ja = csr(jh, c_), csr(ja, c_)
        Ph, Pa = csr(jh, c_, absolute=True), csr(ja, c_, absolute=True)
        kappa[c_] += Ph.T @ (p_h[c_] + q_h[c_].abs()).numpy() + Pa.T @ (p_a[c_] + q_a[c_].abs()).numpy()
        grad[c_] += Jh.T @ (a_h[c_] + q_h[c_]).numpy() + Ja.T @ (a_a[c_] + q_a[c_]).numpy()
        qc = q_c[c_].numpy()[lowi]  # the path through corr_coef: d c / d theta is dense over few components
        kappa[c_] += np.abs(qc).sum() * np.abs(dc_dth[c_])
        grad[c_] += qc.sum() * dc_dth[c_]
    return kappa, lp_scale, grad, lp


def gradient_scale(d: MatchData, theta):
    """Error scale of a float32 evaluation of (lp, d lp / d theta) at ``theta [C, D]``, in float64: returns
    ``(kappa [C, D], lp_scale [C])`` with kappa_i = sum over the elementary terms (and the paths by which they reach
    theta_i) of |d term / d theta_i| and lp_scale = sum of |term| (terms and paths as in ``_gradient_terms``).  A float32 evaluation that rounds each term and each partial sum
    once errs by a small multiple of 2^-24 of these, component by component, however the terms cancel."""
    kappa, lp_scale, _, _ = _gradient_terms(d, theta)
    return kappa, lp_scale


# --------------------------------------------------------------------------------------
# likelihood-only view: what the reference's `_model`s compute from the CONSTRAINED per-team tables
# (checker of bplx_loglik_fwdbwd, the numpyro.factor / custom_vjp route of SURVEY.md 8(b))
# --------------------------------------------------------------------------------------
def likelihood_from_tables(d: MatchData, t: Dict[str, torch.Tensor]):
    """Rates -> Poisson terms -> tau terms from per-team tables ``[..., T]`` (``home_advantage`` ``[...]`` for
    DixonColes), ``confederation_strength [..., Cf]`` and ``corr_coef_raw [...]`` in (0, 1):
    ``dixon_coles.py:63-84``, ``extended_dixon_coles.py:191-246``, ``neutral_dixon_coles.py:236-283``,
    ``neutral_dixon_coles_WC.py:188-232``.  Returns (loglik [...], corr_coef [...])."""
    h, a = _idx(d.home_team), _idx(d.away_team)
    att, dfn = t["attack"], t["defence"]
    dt = att.dtype
    if d.model == "dixon_coles":
        lam_h = torch.exp(att[..., h] - dfn[..., a] + t["home_advantage"][..., None])
        lam_a = torch.exp(att[..., a] - dfn[..., h])
    elif d.model == "extended":
        lam_h = torch.clamp(torch.exp(att[..., h] - dfn[..., a] + t["home_advantage"][..., h]), max=15.0)
        lam_a = torch.clamp(torch.exp(att[..., a] - dfn[..., h]), max=15.0)
    elif d.model in ("neutral", "neutral_wc"):
        n = torch.as_tensor(1 - np.asarray(d.neutral_venue, dtype=np.int64), dtype=dt)
        eta_h = att[..., h] - dfn[..., a] + n * t["home_attack"][..., h] - n * t["away_defence"][..., a]
        eta_a = att[..., a] - dfn[..., h] + n * t["away_attack"][..., a] - n * t["home_defence"][..., h]
        if d.model == "neutral_wc":
            conf = t["confederation_strength"]
            hc, ac = _idx(d.home_conf), _idx(d.away_conf)
            eta_h = eta_h + conf[..., hc] - conf[..., ac]
            eta_a = eta_a + conf[..., ac] - conf[..., hc]
        lam_h, lam_a = torch.exp(eta_h), torch.exp(eta_a)
    else:
        raise ValueError(d.model)
    return _likelihood(d, lam_h, lam_a, t["corr_coef_raw"], dt)
