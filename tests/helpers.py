"""Shared test plumbing: problems, oracle adapters, the CPU plan checker."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from bpl_next_b200 import _abi, data as bdata
from oracle import datasets, models as om

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def to_oracle(arr: bdata.MatchArrays) -> om.MatchData:
    """MatchArrays (product host prep) -> oracle MatchData; covariates are already standardised,
    so the oracle gets them through an identity standardisation (mean 0 / std 1 columns)."""
    cov = None
    if arr.covariates is not None:
        cov = np.asarray(arr.covariates, dtype=np.float64)
    d = om.MatchData(
        model=arr.model, num_teams=arr.num_teams,
        home_team=arr.home_team.astype(np.int64), away_team=arr.away_team.astype(np.int64),
        home_goals=arr.home_goals.astype(np.int64), away_goals=arr.away_goals.astype(np.int64),
        weights=None if arr.weights is None else arr.weights.astype(np.float64),
        neutral_venue=None if arr.neutral_venue is None else arr.neutral_venue.astype(np.int64),
        home_conf=None if arr.home_conf is None else arr.home_conf.astype(np.int64),
        away_conf=None if arr.away_conf is None else arr.away_conf.astype(np.int64),
        num_conferences=arr.num_conferences, covariates=cov,
        gameweek=None if arr.gameweek is None else arr.gameweek.astype(np.int64),
        num_gameweeks=arr.num_gameweeks, walk="as_written" if getattr(arr, "as_written", False) else "intended",
    )
    d.covariates_prestandardised = True
    return d


def small_problem(model: str, seed: int = 0, T: int = 7, M: int = 60, K: int = 0, Cf: int = 3,
                  weighted: bool = True, multi_conf: bool = False, neutral_frac: float = 0.4,
                  low_scores: bool = True) -> bdata.MatchArrays:
    """Random ragged problem with duplicates, missing teams and plenty of low scores."""
    rng = np.random.default_rng(seed)
    h = rng.integers(0, T, M)
    a = (h + rng.integers(1, T, M)) % T if T > 1 else h
    lam = 0.9 if low_scores else 2.0
    hg = rng.poisson(lam, M)
    ag = rng.poisson(lam, M)
    arr = bdata.MatchArrays(model=model, num_teams=T, home_team=h.astype(np.uint16), away_team=a.astype(np.uint16),
                            home_goals=hg.astype(np.uint8), away_goals=ag.astype(np.uint8))
    if weighted and model not in ("dixon_coles", "dynamic"):
        arr.weights = rng.uniform(0.1, 3.0, M).astype(np.float32)
    if model in ("neutral", "neutral_wc"):
        arr.neutral_venue = (rng.random(M) < neutral_frac).astype(np.uint8)
        if arr.weights is None:
            arr.weights = np.ones(M, dtype=np.float32)
    if model == "neutral_wc":
        conf_of = rng.integers(0, Cf, T)
        hc, ac = conf_of[h], conf_of[a]
        if multi_conf:  # a team that changed confederation
            flip = rng.random(M) < 0.15
            hc = np.where(flip, (hc + 1) % Cf, hc)
        arr.home_conf, arr.away_conf, arr.num_conferences = hc.astype(np.uint8), ac.astype(np.uint8), Cf
    if model == "dynamic":
        G = Cf  # (gameweeks travel in the Cf argument)
        arr.neutral_venue = (rng.random(M) < neutral_frac).astype(np.uint8)
        arr.gameweek = rng.integers(0, G, M).astype(np.int32)
        arr.gameweek[0] = G - 1  # make sure the last gameweek exists
        arr.num_gameweeks = G
        arr.weights = None
    if K and model != "dixon_coles":
        X = rng.normal(0, 1, (T, K))
        arr.covariates = ((X - X.mean(0)) / X.std(0)).astype(np.float32)
    return arr


def from_training_data(model, td, epsilon=None, rescale_weights=False):
    return bdata.prepare(model, td, epsilon=epsilon, rescale_weights=rescale_weights)[0]


def random_theta(D, C, seed=0, radius=1.0, dtype=np.float64):
    rng = np.random.default_rng(seed)
    return rng.uniform(-radius, radius, (C, D)).astype(dtype)


# --------------------------------------------------------------------------------------
# per-component error criterion of a float32 log density + gradient (tests/test_gradient_criterion.py calibrates it)
# --------------------------------------------------------------------------------------
EPS32 = 2.0 ** -24
# |g_i - g_o,i| <= CRIT_C * 2^-24 * kappa_i, kappa_i = sum over the elementary terms (and the paths by which they reach
# theta_i) of |d term / d theta_i|; the same with lp and sum |term| (oracle.models.gradient_scale).  The two float32
# restatements of the oracle (closed_form.ClosedForm and models in float32) reach a gradient ratio of 163 (configs[2]
# data at radius 2: a confederation strength, a sum over 40,000 matches) and an lp ratio of 32 on the cases of
# tests/test_gradient_criterion.py.  CRIT_C is about three times the larger.
CRIT_C = 512.0


def criterion_ratios(d: om.MatchData, theta64, lp, grad, ref=None):
    """(|lp - lp_o| / (2^-24 sum |term|) [C], |g - g_o| / (2^-24 kappa) [C, D]) against the float64 oracle;
    ``ref`` = (lp_o, g_o, kappa, lp_scale) when the caller has them."""
    if ref is None:
        lp_o, g_o, _ = om.log_density_and_grad(d, theta64)
        kappa, lp_scale = om.gradient_scale(d, theta64)
    else:
        lp_o, g_o, kappa, lp_scale = ref
    with np.errstate(divide="ignore", invalid="ignore"):
        rg = np.abs(np.asarray(grad, np.float64) - g_o) / (EPS32 * kappa)
        rl = np.abs(np.asarray(lp, np.float64) - lp_o) / (EPS32 * lp_scale)
    rg[(kappa == 0) & (np.asarray(grad) == g_o)] = 0.0  # a component no term depends on (K = 0 sites are absent)
    return rl, rg


def criterion_failures(d: om.MatchData, theta64, lp, grad, c: float = CRIT_C, limit: int = 8, ref=None):
    """Components that break the criterion, as 'chain c: site[index] ratio r' (worst first); [] when it holds."""
    rl, rg = criterion_ratios(d, theta64, lp, grad, ref)
    names = []
    for name, shape, _ in om.site_layout(d.model, d.num_teams, d.num_covariates,
                                         d.num_conferences if d.model == "neutral_wc" else 0, d.num_gameweeks):
        n = int(np.prod(shape)) if shape else 1
        names += [name] if shape == () else [f"{name}{list(np.unravel_index(i, shape))}" for i in range(n)]
    out = [(r, f"chain {ch}: lp ratio {r:.3g}") for ch, r in enumerate(rl) if not r <= c]
    bad = np.argwhere(~(rg <= c))
    out += [(rg[ch, i], f"chain {ch}: {names[i]} ratio {rg[ch, i]:.3g}") for ch, i in bad]
    out.sort(key=lambda x: -x[0] if np.isfinite(x[0]) else -np.inf)
    return [s for _, s in out[:limit]] + ([f"... {len(out) - limit} more"] if len(out) > limit else [])


def assert_criterion(d: om.MatchData, theta64, lp, grad, what: str = "", ref=None):
    bad = criterion_failures(d, theta64, lp, grad, ref=ref)
    assert not bad, f"{what}: per-component criterion (c = {CRIT_C:g}) fails: " + "; ".join(bad)


# --------------------------------------------------------------------------------------
_plancheck = None


def plancheck_lib():
    global _plancheck
    if _plancheck is None:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
        lib = C.CDLL(os.path.join(ROOT, "oracle", "_build", "libplancheck.so"))
        lib.bplx_plancheck_eval.argtypes = [C.POINTER(_abi.ProblemDesc), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_char_p, C.c_int]
        lib.bplx_plancheck_eval.restype = C.c_int
        lib.bplx_plancheck_eval2.argtypes = [C.POINTER(_abi.ProblemDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_char_p, C.c_int]
        lib.bplx_plancheck_eval2.restype = C.c_int
        _plancheck = lib
    return _plancheck


def plancheck_eval(arr: bdata.MatchArrays, theta: np.ndarray, split_idx: int = 0):
    """Double-precision walk of the product's static plan (for 2**split_idx CTAs per chain group), chain by chain."""
    lib = plancheck_lib()
    desc = arr.desc()
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    Cn, D = theta.shape
    lp = np.zeros(Cn)
    grad = np.zeros((Cn, D))
    cc = np.zeros(Cn)
    err = C.create_string_buffer(512)
    for c in range(Cn):
        one_lp, one_cc = C.c_double(), C.c_double()
        rc = lib.bplx_plancheck_eval2(C.byref(desc), split_idx, theta[c].ctypes.data, C.addressof(one_lp),
                                      grad[c].ctypes.data, C.addressof(one_cc), err, 512)
        if rc != 0:
            raise RuntimeError(f"plancheck rc={rc}: {err.value.decode()}")
        lp[c], cc[c] = one_lp.value, one_cc.value
    return lp, grad, cc
