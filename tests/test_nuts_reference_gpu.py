"""GPU: the NUTS step kernel (csrc/nuts.cu) transition by transition against the float64 reference sampler
(oracle/nuts.py), which consumes the same Philox random numbers.  Every launch branch (both state layouts, every
register-resident geometry, the stage-by-stage kernel) at a fixed step size, deep trees, the depth limit, divergent and
non-finite leaves, thinning / row pitch / chain offsets, and the models' own log-density kernel.

A chain matches when every stored draw, lp and acceptance statistic, its leapfrog / divergence / transition counts, its
final step size and its inverse mass agree with the reference within tolerance.  A float32 sampler may take a
different branch where the reference's decision margin is tiny: such a chain is excused when the reference recorded a
margin below ``tau`` at or before the first transition that differs -- and no more than 5 % of the chains may be."""
from dataclasses import dataclass

import numpy as np
import pytest

from bpl_next_b200 import nuts as bn
from oracle import nuts as on

pytestmark = pytest.mark.gpu


@dataclass
class Tol:
    draw: float = 1e-4    # x (sd_d + |mean_d|) of the reference draws
    lp: float = 1e-5      # x (1 + |lp|)
    accept: float = 1e-4  # (measured on a B200 up to 2.5e-5 at D = 300: dH is a difference of float32 energies)
    rel: float = 1e-4     # step size and inverse mass, relative
    tau: float = 1e-4     # decision margin below which a different branch is excused

    def times(self, f):
        return Tol(self.draw * f, self.lp * f, self.accept * f, self.rel * f, self.tau * f)


GAUSS = Tol()
K1 = GAUSS.times(10.0)  # the log-density kernel's gradient carries a 1e-4 relative error


def _compare(name, run, ref, chains, cfg, tol):
    """Chain by chain; returns the summary line, raises with the chain, the transition and the reference's decisions
    there on any mismatch the reference's margins do not excuse."""
    S = run.samples.detach().cpu().numpy().astype(np.float64)  # [K, D, C]
    LP = run.lp.detach().cpu().numpy().astype(np.float64)
    AC = run.accept.detach().cpu().numpy().astype(np.float64)
    IM = run.inv_mass.detach().cpu().numpy().astype(np.float64)
    R = np.stack([r.samples for r in ref])  # [n, K, D]
    scale = R.std(axis=(0, 1)) + np.abs(R.mean(axis=(0, 1)))
    worst = dict(draw=0.0, lp=0.0, accept=0.0, step=0.0, inv_mass=0.0)
    excused, failures = [], []
    for i, c in enumerate(chains):
        r = ref[i]
        e_draw = (np.abs(S[:, :, c] - r.samples) / scale).max(axis=1)
        e_lp = np.abs(LP[:, c] - r.lp) / (1 + np.abs(r.lp))
        e_acc = np.abs(AC[:, c] - r.accept)
        e_step = abs(run.step_size[c] / r.step_size - 1)
        e_im = (np.abs(IM[:, c] - r.inv_mass) / r.inv_mass).max()
        bad = np.flatnonzero(~((e_draw <= tol.draw) & (e_lp <= tol.lp) & (e_acc <= tol.accept)))  # NaN is bad
        counts = (int(run.num_leapfrog[c]), int(run.num_divergent[c]), int(run.transitions[c]))
        want = (r.num_leapfrog, r.num_divergent, r.transitions)
        # After a different branch the two samplers consume different launches, so every later draw differs: the first
        # difference lies between the last stored draw that agrees and the first that does not (or the end of the run
        # when only the counts, the step size or the inverse mass differ).
        stored = [cfg.num_warmup + k * cfg.thin for k in range(len(r.lp))]
        what = None
        if len(bad):
            k = bad[0]
            lo, hi = (stored[k - 1] if k else 0), stored[k]
            what = (f"draw {k}: error {e_draw[k]:.2e} x scale, lp error {e_lp[k]:.2e}, accept {AC[k, c]:.6f} vs "
                    f"{r.accept[k]:.6f}")
        elif counts != want or not (e_step <= tol.rel and e_im <= tol.rel):
            lo, hi = (stored[-1] if stored else 0), r.transitions - 1
            what = (f"(leapfrogs, divergences, transitions) {counts} vs {want}, step size {run.step_size[c]:.7g} vs "
                    f"{r.step_size:.7g}, inverse mass error {e_im:.2e}")
        if what is None:
            for key, v in (("draw", e_draw.max(initial=0)), ("lp", e_lp.max(initial=0)),
                           ("accept", e_acc.max(initial=0)), ("step", e_step), ("inv_mass", e_im)):
                worst[key] = max(worst[key], float(v))
            continue
        margin = r.min_margin(lo, hi)
        if margin < tol.tau:
            excused.append(c)
        else:
            t = min(range(lo, hi + 1), key=lambda tt: r.min_margin(tt, tt))
            failures.append(f"chain {c}, first difference at transitions {lo}..{hi} (smallest margin there "
                            f"{margin:.2e}, at transition {t}, {r.leapfrogs[t]} reference leapfrogs): {what}\n"
                            f"    reference decisions at transition {t}: {r.history(t)[:1500]}")
    n = len(chains)
    line = (f"[nuts-ref] {name}: {n - len(excused) - len(failures)}/{n} matched, {len(excused)} excused, worst "
            + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    print(line)
    assert not failures, f"{name}: {len(failures)} of {n} chains differ from the reference:\n" + "\n".join(failures[:5])
    assert len(excused) <= 0.05 * n, f"{name}: {len(excused)} of {n} chains excused by small margins: {excused}"
    return line


def _run(name, target, theta0, cfg, tol=GAUSS, layout="chain_minor", chains=None, pad_rows=False):
    """GPU run from theta0 [C, D] (float32) and the reference on `chains` (all by default)."""
    import torch

    potential, potential_cm, ref_potential = target
    C = theta0.shape[0]
    chains = list(range(C)) if chains is None else list(chains)
    run = bn.sample(potential, torch.from_numpy(np.ascontiguousarray(theta0.T)).cuda(), num_warmup=cfg.num_warmup,
                    num_samples=cfg.num_samples, thin=cfg.thin, seed=cfg.seed, max_tree_depth=cfg.max_tree_depth,
                    step_size=cfg.step_size, chain_offset=cfg.chain_offset, pad_rows=pad_rows,
                    potential_cm=potential_cm if layout == "chain_major" else None, state_layout=layout)
    ref = on.sample(ref_potential, theta0[chains].astype(np.float64), cfg, chains)
    _compare(name, run, ref, chains, cfg, tol)
    return run, ref


def _target(lp_fn):
    """(potential [D, C], potential_cm [C, D], reference potential) from a torch function theta [C, D] -> lp [C]; the
    gradient by autograd (float32 on the GPU, float64 for the reference)."""
    import torch

    def ev(theta):  # [C, D]
        th = theta.detach().clone().requires_grad_(True)
        lp = lp_fn(th)
        (g,) = torch.autograd.grad(lp.sum(), th)
        return lp.detach(), g

    def potential(theta, lp, grad):
        a, g = ev(theta.t())
        lp.copy_(a)
        grad.copy_(g.t())

    def potential_cm(theta, lp, grad):
        a, g = ev(theta)
        lp.copy_(a)
        grad.copy_(g)

    def ref_potential(theta):
        a, g = ev(torch.from_numpy(theta))
        return a.numpy(), g.numpy()

    return potential, potential_cm, ref_potential


def _gauss(D, seed, spread=0.5):
    """Independent normals, sd in exp([-spread, spread]); mu, sd as float32 values on both sides."""
    import torch

    rng = np.random.default_rng(seed)
    mu = rng.uniform(-1, 1, D).astype(np.float32)
    sd = np.exp(rng.uniform(-spread, spread, D)).astype(np.float32)

    consts = {}  # per device / dtype, made outside any CUDA-graph capture (the first, eager block)

    def lp_fn(th):
        key = (th.device, th.dtype)
        if key not in consts:
            consts[key] = tuple(torch.as_tensor(v, device=th.device, dtype=th.dtype) for v in (mu, sd))
        m, s = consts[key]
        z = (th - m) / s
        return -0.5 * (z * z).sum(1)

    def init(C, radius=1.5):
        return (mu + sd * rng.uniform(-radius, radius, (C, D))).astype(np.float32)

    return _target(lp_fn), init


# D -> the launch branch it selects: chain-minor <32,4> (D <= 64), <16,4> (D <= 128), <8,4> (D <= 256), generic;
# chain-major <8,2,true> (D <= 64), <8,4,true> (D <= 128), generic
@pytest.mark.parametrize("layout,D,generic", [
    ("chain_minor", 6, False), ("chain_minor", 44, False), ("chain_minor", 64, False), ("chain_minor", 100, False),
    ("chain_minor", 200, False), ("chain_minor", 300, False), ("chain_major", 44, False), ("chain_major", 113, False),
    ("chain_major", 300, False), ("chain_minor", 44, True), ("chain_major", 113, True)])
def test_fixed_step_transitions_match_reference(layout, D, generic, bplx_env):
    """No warm-up, a fixed step: 70 chains (not a multiple of any block's chain count), 40 draws each."""
    bplx_env(BPLX_NUTS_GENERIC="1" if generic else None)
    target, init = _gauss(D, D)
    cfg = on.Config(num_warmup=0, num_samples=40, seed=11, step_size=0.25, max_tree_depth=6)
    _, ref = _run(f"fixed {layout} D={D}{' generic' if generic else ''}", target, init(70), cfg, layout=layout)
    assert sum(r.early_subtree_turns for r in ref) + sum(r.rejected_merges for r in ref) > 0


@pytest.mark.parametrize("layout,D,generic", [("chain_minor", 6, False), ("chain_major", 44, False),
                                              ("chain_minor", 6, True), ("chain_major", 44, True)])
def test_warmup_adaptation_matches_reference(layout, D, generic, bplx_env):
    """20 warm-up steps are three windows, (0, 2), (3, 17), (18, 19): dual averaging from the initial step, Welford
    over the middle window, its end (regularised variance -> inverse mass, the step-size search restarted around
    10 eps) and exp(x_avg) after the last step.  Each chain's adapted step size and inverse mass against the reference.

    Warm-up amplifies float32 rounding: dual averaging multiplies acceptance errors (~1e-5 at a fixed step) by
    sqrt(t) / gamma, and the restart after the window end weighs the last two steps alone.  Measured on a B200: step
    sizes up to 1.9 % apart, inverse masses 4.7 %, and branches taken differently at margins up to 2e-2 -- so draws are
    not compared here, and up to 10 % of the chains may be excused.  Dropping Stan's regularisation moves the inverse mass by 25 %, exp(x) for exp(x_avg) the step
    by far more than 5 %."""
    bplx_env(BPLX_NUTS_GENERIC="1" if generic else None)
    target, init = _gauss(D, 100 + D, spread=1.0)
    cfg = on.Config(num_warmup=20, num_samples=1, seed=5, step_size=0.5, max_tree_depth=7)
    assert on.adaptation_schedule(20) == [(0, 2), (3, 17), (18, 19)]
    import torch

    theta0 = init(70)
    run = bn.sample(target[0], torch.from_numpy(np.ascontiguousarray(theta0.T)).cuda(), num_warmup=20, num_samples=1,
                    seed=5, step_size=0.5, max_tree_depth=7, potential_cm=target[1] if layout == "chain_major" else None,
                    state_layout=layout)
    ref = on.sample(target[2], theta0.astype(np.float64), cfg)
    IM = run.inv_mass.detach().cpu().numpy().astype(np.float64)
    e_step = np.array([abs(run.step_size[c] / r.step_size - 1) for c, r in enumerate(ref)])
    e_im = np.array([(np.abs(IM[:, c] - r.inv_mass) / r.inv_mass).max() for c, r in enumerate(ref)])
    assert (run.transitions == 21).all()
    bad = np.flatnonzero(~((e_step <= 5e-2) & (e_im <= 5e-2)))
    excused = [c for c in bad if ref[c].min_margin(0, 19) < 2e-2]
    ok = np.setdiff1d(np.arange(70), bad)
    print(f"[nuts-ref] warm-up 20 {layout} D={D}{' generic' if generic else ''}: {len(ok)}/70 matched, "
          f"{len(excused)} excused, worst step {e_step[ok].max():.2e}, inv_mass {e_im[ok].max():.2e}")
    failures = [f"chain {c}: step size {run.step_size[c]:.7g} vs {ref[c].step_size:.7g}, inverse mass error {e_im[c]:.2e}, "
                f"smallest warm-up margin {ref[c].min_margin(0, 19):.2e}" for c in bad if c not in excused]
    assert not failures, "\n".join(failures[:5])
    # (measured on a B200: 4 of 70 at D = 44; with either mutation above, 67 or more)
    assert len(excused) <= 0.1 * 70, f"{len(excused)} of 70 chains excused by small margins: {excused}"


def test_finite_divergences_match_reference():
    """A Gaussian with one sd of 0.12 at step 0.3: the leapfrog is unstable along it (step > 2 sd) and dH passes
    max_delta_energy = 1000 in many transitions while the log-density stays finite."""
    sd = np.array([0.12, 1, 1, 1, 1, 1], dtype=np.float32)
    target = _target(lambda th: -0.5 * ((th / torch_like(th, sd)) ** 2).sum(1))
    rng = np.random.default_rng(9)
    theta0 = (sd * rng.normal(size=(70, 6))).astype(np.float32)
    cfg = on.Config(num_warmup=0, num_samples=10, seed=9, step_size=0.3, max_tree_depth=6)
    # (the unstable direction grows rounding errors 2.5-fold per leapfrog, and from draw to draw: measured on a B200 up
    # to 4e-3 x scale in 10 draws, 2e-2 in 30)
    run, ref = _run("finite divergences", target, theta0, cfg, tol=GAUSS.times(100.0))
    assert sum(r.divergences for r in ref) > 0 and sum(r.nonfinite_leaves for r in ref) == 0
    assert run.num_divergent.sum() > 0


_CONSTS = {}


def torch_like(th, v):
    """The float32 constants ``v`` as a tensor on ``th``'s device and dtype, made once (outside CUDA-graph capture)."""
    import torch

    key = (id(v), th.device, th.dtype)
    if key not in _CONSTS:
        _CONSTS[key] = torch.as_tensor(v, device=th.device, dtype=th.dtype)
    return _CONSTS[key]


@pytest.mark.parametrize("generic", [False, True])
def test_deep_trees_match_reference(generic, bplx_env):
    """A unit Gaussian at step 0.05: subtrees of 32 and more leaves, whose last leaves are tested against 5 and 6
    checkpoint levels (the stage-by-stage kernel's second pass of U-turn slots)."""
    bplx_env(BPLX_NUTS_GENERIC="1" if generic else None)
    target = _target(lambda th: -0.5 * (th * th).sum(1))
    rng = np.random.default_rng(1)
    cfg = on.Config(num_warmup=0, num_samples=8, seed=2, step_size=0.05, max_tree_depth=8)
    _, ref = _run(f"deep trees{' generic' if generic else ''}", target, rng.normal(size=(32, 6)).astype(np.float32), cfg)
    assert max(r.max_trailing_ones for r in ref) >= 5


@pytest.mark.parametrize("depth,step,C,N", [(1, 0.3, 64, 40), (12, 0.0005, 8, 2)])
def test_depth_limit_matches_reference(depth, step, C, N):
    """The smallest and the largest max_tree_depth: trajectories that stop at the limit (4,096 leaves at depth 12)."""
    target = _target(lambda th: -0.5 * (th * th).sum(1))
    rng = np.random.default_rng(depth)
    cfg = on.Config(num_warmup=0, num_samples=N, seed=3, step_size=step, max_tree_depth=depth)
    _, ref = _run(f"max_tree_depth={depth}", target, rng.normal(size=(C, 6)).astype(np.float32), cfg)
    assert sum(r.depth_limit_hits for r in ref) > 0


def test_non_finite_log_density_matches_reference():
    """A Gaussian whose log-density is -inf on one half-space and NaN on another: those leaves are rejected and end
    their trajectory as divergent."""
    import torch

    def lp_fn(th):
        lp = -0.5 * (th * th).sum(1)
        lp = torch.where(th[:, 0] > 1.0, torch.full_like(lp, -float("inf")), lp)
        return torch.where(th[:, 1] < -1.2, torch.full_like(lp, float("nan")), lp)

    rng = np.random.default_rng(4)
    cfg = on.Config(num_warmup=0, num_samples=30, seed=4, step_size=0.3, max_tree_depth=6)
    run, ref = _run("non-finite", _target(lp_fn), rng.uniform(-0.8, 0.8, (70, 6)).astype(np.float32), cfg)
    assert sum(r.nonfinite_leaves for r in ref) > 0 and run.num_divergent.sum() > 0


def test_thinning_row_pitch_and_chain_offset():
    """thin = 3, a padded row pitch (1,024 chains: ld = 1,056) and chain_offset = 37, against the reference on every
    16th chain; and chains [k, C) run on their own with chain_offset + k are the same chains of the full run, bit for
    bit (what a rank of a multi-GPU fit does)."""
    import torch

    target, init = _gauss(6, 7)
    theta0 = init(1024)
    cfg = on.Config(num_warmup=0, num_samples=10, thin=3, seed=8, step_size=0.25, max_tree_depth=6, chain_offset=37)
    run, _ = _run("thin / pitch / offset", target, theta0, cfg, chains=range(0, 1024, 16), pad_rows=True)
    assert run.samples.shape == (4, 6, 1024)
    k = 300
    part = bn.sample(target[0], torch.from_numpy(np.ascontiguousarray(theta0[k:].T)).cuda(), num_warmup=0,
                     num_samples=10, thin=3, seed=8, max_tree_depth=6, step_size=0.25, chain_offset=37 + k)
    assert torch.equal(part.samples, run.samples[:, :, k:]) and torch.equal(part.lp, run.lp[:, k:])
    assert torch.equal(part.accept, run.accept[:, k:])
    assert np.array_equal(part.num_leapfrog, run.num_leapfrog[k:])


@pytest.mark.parametrize("model,layout", [("dixon_coles", "chain_minor"), ("dixon_coles", "chain_major"),
                                          ("extended", "chain_minor"), ("extended", "chain_major"),
                                          ("neutral_wc", "chain_major")])
def test_models_match_reference(model, layout):
    """The production path: the log-density kernel + the NUTS step on the reference's dummy leagues, against the
    reference driven by the float64 oracle density.  64 chains near the prior's centre, a small fixed step, 10 draws.
    (With warm-up these chains leave the tolerances: the models' curvature at the first, large step sizes amplifies
    the step-size differences the Gaussian warm-up cases bound.)"""
    from bpl_next_b200 import Problem
    from oracle import datasets, models as om
    from tests import helpers as H

    if model == "neutral_wc":
        arr = H.from_training_data(model, datasets.neutral_dummy_data(), epsilon=0.2)
    else:
        arr = H.from_training_data(model, datasets.dummy_data())
    p = Problem(arr)
    d = H.to_oracle(arr)

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    def potential_cm(theta, lp, grad):
        p.logdensity(theta, chain_minor=False, lp=lp, grad=grad)

    def ref_potential(theta):
        lp, g, _ = om.log_density_and_grad(d, theta)
        return lp, g

    rng = np.random.default_rng(3)
    theta0 = rng.uniform(-0.1, 0.1, (64, p.D)).astype(np.float32)
    cfg = on.Config(num_warmup=0, num_samples=10, seed=12, step_size=0.01, max_tree_depth=5)
    _run(f"{model} {layout} D={p.D}", (potential, potential_cm, ref_potential), theta0, cfg, tol=K1, layout=layout)
    p.close()
