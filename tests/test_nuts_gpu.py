"""GPU: the batched NUTS transition (bplx_nuts_step) on targets with known answers, and on the Dixon-Coles kernel."""
import numpy as np
import pytest

from bpl_next_b200 import nuts as bn

pytestmark = pytest.mark.gpu


def test_adaptation_schedule_matches_numpyro_defaults():
    assert bn.adaptation_schedule(500) == [(0, 74), (75, 99), (100, 149), (150, 249), (250, 449), (450, 499)]
    assert bn.adaptation_schedule(10) == [(0, 9)]
    s = bn.adaptation_schedule(100)
    assert s[0] == (0, 14) and s[-1] == (90, 99) and s[1][0] == 15 and s[-2][1] == 89


def test_gaussian_target_moments():
    """Independent normals with very different scales: means / sds must come out within Monte-Carlo error."""
    import torch
    from bpl_next_b200 import diagnostics as dg

    D, C = 6, 512
    mu = torch.tensor([0.0, 1.0, -2.0, 3.0, 0.5, -0.5], device="cuda")[:, None]
    sd = torch.tensor([1.0, 0.1, 10.0, 2.0, 0.5, 5.0], device="cuda")[:, None]

    def potential(theta, lp, grad):
        z = (theta - mu) / sd
        lp.copy_(-0.5 * (z * z).sum(0))
        grad.copy_(-z / sd)

    g = torch.Generator(device="cuda").manual_seed(0)
    theta0 = (torch.rand((D, C), generator=g, device="cuda") * 4 - 2)
    run = bn.sample(potential, theta0, num_warmup=300, num_samples=200, seed=1)
    x = run.samples.double()  # [N, D, C]
    mean = x.mean(dim=(0, 2)).cpu().numpy()
    std = x.permute(1, 0, 2).reshape(D, -1).std(dim=1).cpu().numpy()
    ess = dg.effective_sample_size(run.samples).cpu().numpy()
    assert ess.min() > 5000, ess
    mcse = sd[:, 0].cpu().numpy() / np.sqrt(ess)
    assert np.all(np.abs(mean - mu[:, 0].cpu().numpy()) < 5 * mcse), (mean, mcse)
    np.testing.assert_allclose(std, sd[:, 0].cpu().numpy(), rtol=0.03)
    rhat = dg.split_rhat(run.samples).cpu().numpy()
    assert np.all(rhat < 1.02), rhat
    assert run.num_divergent.sum() == 0
    # the adapted inverse mass matrix is the posterior variance (diagonal), chain by chain
    imm = run.inv_mass.mean(dim=1).cpu().numpy()
    np.testing.assert_allclose(imm, (sd[:, 0] ** 2).cpu().numpy(), rtol=0.35)
    assert 0.6 < run.accept.mean().item() < 0.95


def test_dixon_coles_posterior_is_stationary_across_seeds():
    """Two independent runs on the reference's dummy league agree within Monte-Carlo error, and the chains mix."""
    import torch
    from bpl_next_b200 import Problem, diagnostics as dg
    from oracle import datasets
    from tests import helpers as H

    arr = H.from_training_data("dixon_coles", datasets.dummy_data())
    p = Problem(arr)
    C = 256

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    means = []
    for seed in (3, 4):
        g = torch.Generator(device="cuda").manual_seed(seed)
        theta0 = torch.rand((p.D, C), generator=g, device="cuda") * 4 - 2  # init_to_uniform(radius=2)
        run = bn.sample(potential, theta0, num_warmup=300, num_samples=150, seed=seed)
        assert dg.split_rhat(run.samples).max().item() < 1.05
        ess = dg.effective_sample_size(run.samples)
        sd = run.samples.permute(1, 0, 2).reshape(p.D, -1).std(dim=1)
        means.append((run.samples.double().mean(dim=(0, 2)), sd.double() / ess.sqrt()))
        assert run.num_divergent.mean() < 1.0
    diff = (means[0][0] - means[1][0]).abs()
    tol = 6 * torch.sqrt(means[0][1] ** 2 + means[1][1] ** 2)
    assert bool((diff < tol).all()), (diff / tol).max().item()
    # home advantage posterior mean: log(782/645) ~ 0.19 is the data's home/away goal ratio (prior N(0.1, 0.2))
    ha = means[0][0][0].item()
    assert 0.1 < ha < 0.3, ha


@pytest.mark.parametrize("layout", ["chain_minor", "chain_major"])
@pytest.mark.parametrize("D,C", [(6, 70), (44, 96), (64, 33), (113, 21)])
def test_register_resident_step_matches_stage_by_stage_kernel(D, C, layout, bplx_env):
    """Small models run the NUTS bookkeeping out of registers (nuts_step_fast_kernel); with the same block geometry it
    does the same arithmetic in the same order as the stage-by-stage kernel, so whole runs must agree bit for bit:
    draws, acceptance statistics, leapfrog counts, adapted step sizes and mass matrices.  Both state layouts (chain-minor:
    lane = chain, up to 16 slices; chain-major: a warp per chain, D <= 128)."""
    import torch

    if layout == "chain_minor" and D > 64:
        pytest.skip("chain-minor: the two kernels share their geometry up to D = 64 only")

    g = torch.Generator(device="cuda").manual_seed(3)
    sd = torch.exp(torch.rand((D, 1), generator=g, device="cuda") * 3 - 1.5)
    mu = torch.rand((D, 1), generator=g, device="cuda") * 2 - 1

    def potential(theta, lp, grad):
        z = (theta - mu) / sd
        lp.copy_(-0.5 * (z * z).sum(0))
        grad.copy_(-z / sd)

    def potential_cm(theta, lp, grad):
        z = (theta - mu[:, 0]) / sd[:, 0]
        lp.copy_(-0.5 * (z * z).sum(1))
        grad.copy_(-z / sd[:, 0])

    theta0 = torch.rand((D, C), generator=g, device="cuda") * 4 - 2
    runs = []
    for generic in (False, True):
        bplx_env(BPLX_NUTS_GENERIC="1" if generic else None)
        runs.append(bn.sample(potential, theta0.clone(), num_warmup=120, num_samples=40, seed=7, use_graph=False,
                              potential_cm=potential_cm, state_layout=layout))
    a, b = runs
    assert a.launches == b.launches
    assert torch.equal(a.samples, b.samples)
    assert torch.equal(a.lp, b.lp) and torch.equal(a.accept, b.accept)
    assert torch.equal(a.inv_mass, b.inv_mass)
    assert np.array_equal(a.step_size, b.step_size) and np.array_equal(a.num_leapfrog, b.num_leapfrog)


@pytest.mark.parametrize("D", [100, 200])
def test_register_resident_step_wide_geometries(D):
    """64 < D <= 256 uses 16 or 8 chains per block (32 / 64 slices per chain): no bit-twin to compare with, so the
    moments of a Gaussian target are checked."""
    import torch
    from bpl_next_b200 import diagnostics as dg

    C = 200
    g = torch.Generator(device="cuda").manual_seed(5)
    sd = torch.exp(torch.rand((D, 1), generator=g, device="cuda") * 2 - 1)
    mu = torch.rand((D, 1), generator=g, device="cuda") * 2 - 1

    def potential(theta, lp, grad):
        z = (theta - mu) / sd
        lp.copy_(-0.5 * (z * z).sum(0))
        grad.copy_(-z / sd)

    theta0 = torch.rand((D, C), generator=g, device="cuda") * 4 - 2
    run = bn.sample(potential, theta0, num_warmup=300, num_samples=100, seed=2)
    x = run.samples.double()
    mean = x.mean(dim=(0, 2))
    std = x.permute(1, 0, 2).reshape(D, -1).std(dim=1)
    ess = dg.effective_sample_size(run.samples)
    mcse = sd[:, 0].double() / ess.double().sqrt()
    assert float(((mean - mu[:, 0].double()).abs() / mcse).max()) < 5.5
    assert float((std / sd[:, 0].double() - 1).abs().max()) < 0.06
    assert run.num_divergent.sum() == 0


def test_runs_are_reproducible_with_the_dixon_coles_kernel():
    """Same data, seed and chain count -> the same draws, bit for bit (no timing-dependent arithmetic anywhere between
    the log-density kernel and the NUTS step; regression test for the arg-max tie race far from the typical set)."""
    import torch
    from bpl_next_b200 import Problem
    from oracle import datasets
    from tests import helpers as H

    arr = H.from_training_data("dixon_coles", datasets.dummy_data())
    p = Problem(arr)
    g = torch.Generator(device="cuda").manual_seed(11)
    theta0 = torch.rand((p.D, 96), generator=g, device="cuda") * 4 - 2

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    a = bn.sample(potential, theta0.clone(), num_warmup=60, num_samples=20, seed=1)
    b = bn.sample(potential, theta0.clone(), num_warmup=60, num_samples=20, seed=1, use_graph=False)
    assert a.launches == b.launches
    assert torch.equal(a.samples, b.samples) and torch.equal(a.lp, b.lp)
    assert np.array_equal(a.num_leapfrog, b.num_leapfrog)
    p.close()


def test_dependent_launch_does_not_change_results(bplx_env):
    """K1 and the NUTS step start their preambles before the previous kernel of the stream has finished (programmatic
    dependent launch).  Anything read too early would show up as a different run: with and without it, eager and as a
    CUDA graph, the draws must be identical."""
    import torch
    from bpl_next_b200 import Problem
    from oracle import datasets
    from tests import helpers as H

    arr = H.from_training_data("extended", datasets.dummy_data())
    p = Problem(arr)
    g = torch.Generator(device="cuda").manual_seed(5)
    theta0 = torch.rand((p.D, 160), generator=g, device="cuda") * 4 - 2

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    runs = []
    for no_pdl in (False, True):
        bplx_env(BPLX_NO_PDL="1" if no_pdl else None)
        for graph in (True, False):
            runs.append(bn.sample(potential, theta0.clone(), num_warmup=50, num_samples=15, seed=3, use_graph=graph))
    for r in runs[1:]:
        assert r.launches == runs[0].launches
        assert torch.equal(r.samples, runs[0].samples) and torch.equal(r.lp, runs[0].lp)
    p.close()


@pytest.mark.parametrize("model", ["dixon_coles", "extended", "neutral_wc"])
def test_posterior_matches_independent_cpu_sampler(model):
    """Posterior means and spreads of a GPU fit (K1 + the NUTS kernel) against tests/golden/posterior_<model>.npz:
    plain HMC on the float64 CPU oracle density, an independent sampler sharing no code with the CUDA path
    (scripts/make_posterior_golden.py; R-hat <= 1.01, ESS >= 1e4 there).  Every component must agree within 5 combined
    Monte-Carlo standard errors -- BASELINE.json: "posterior means and quantiles within Monte-Carlo standard error"."""
    import os
    import torch
    from bpl_next_b200 import Problem, diagnostics as dg
    from oracle import datasets
    from tests import helpers as H

    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", f"posterior_{model}.npz"))
    if model in ("dixon_coles", "extended"):
        arr = H.from_training_data(model, datasets.dummy_data())
    else:
        arr = H.from_training_data("neutral_wc", datasets.neutral_dummy_data(), epsilon=0.2)
    p = Problem(arr)
    C = 512
    g = torch.Generator(device="cuda").manual_seed(21)
    theta0 = torch.rand((p.D, C), generator=g, device="cuda") * 4 - 2

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    # (the confederation strengths mix slowly: more draws per chain there)
    run = bn.sample(potential, theta0, num_warmup=400, num_samples=120 if model == "dixon_coles" else 300, seed=9)
    x = run.samples  # [N, D, C] unconstrained
    lay = p.layout

    def site(name):
        o, n, _ = lay[name]
        return x[:, o:o + n, :]

    std_a, std_d = torch.exp(site("std_attack")), torch.exp(site("std_defence"))
    N = x.shape[0]
    flat = x.permute(0, 2, 1).reshape(N * C, p.D).contiguous()
    cc = p.logdensity(flat)[2].reshape(N, C)[:, None, :]
    if model == "dixon_coles":
        q = {"attack": std_a * site("attack_decentered"), "defence": site("mean_defence") + std_d * site("defence_decentered"),
             "home_advantage": site("home_advantage")}
    elif model == "extended":
        q = {"attack": std_a * site("standardised_attack"), "defence": site("mean_defence") + std_d * site("standardised_defence"),
             "home_advantage": site("mean_home_advantage") + torch.exp(site("std_home_advantage")) * site("home_advantage_decentered"),
             "rho": 2.0 * torch.sigmoid(site("u")) - 1.0}
    else:
        q = {"attack": std_a * site("standardised_attack"), "defence": site("mean_defence") + std_d * site("standardised_defence"),
             "confederation_strength": site("confederation_strength_decentered")}
        for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
            q[nm] = site("mean_" + nm) + torch.exp(site("std_" + nm)) * site(nm + "_decentered")
    q.update({"std_attack": std_a, "std_defence": std_d, "corr_coef": cc})
    assert float(dg.split_rhat(x).max()) < 1.05
    for k, v in q.items():
        ess = dg.effective_sample_size(v.contiguous()).double().cpu().numpy()
        mean = v.double().mean(dim=(0, 2)).cpu().numpy()
        sd = v.double().permute(1, 0, 2).reshape(v.shape[1], -1).std(dim=1).cpu().numpy()
        mcse = np.sqrt((sd / np.sqrt(ess)) ** 2 + gold[k + "_mcse"] ** 2)
        z = np.abs(mean - gold[k + "_mean"]) / mcse
        assert z.max() < 5.0, (k, z.max(), mean, gold[k + "_mean"])
        np.testing.assert_allclose(sd, gold[k + "_sd"], rtol=0.08, err_msg=k)
    p.close()


def _gauss(D, seed):
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    mu = torch.randn((D, 1), generator=g, device="cuda") * 2
    sd = torch.exp(0.7 * torch.randn((D, 1), generator=g, device="cuda"))

    def potential(theta, lp, grad):  # [D, C]
        z = (theta - mu) / sd
        lp.copy_(-0.5 * (z * z).sum(0))
        grad.copy_(-z / sd)

    def potential_cm(theta, lp, grad):  # [C, D] (padded row pitch)
        z = (theta - mu[:, 0]) / sd[:, 0]
        lp.copy_(-0.5 * (z * z).sum(1))
        grad.copy_(-z / sd[:, 0])

    return mu, sd, potential, potential_cm, g


def test_chain_major_state_samples_the_same_target():
    """state_layout='chain_major' (a warp per chain, [C, D] vectors): means / sds of independent normals within Monte-Carlo
    error, the adapted inverse mass is the variance, streaming accumulators equal their specification."""
    import torch
    from bpl_next_b200 import diagnostics as dg

    D, C = 300, 256
    mu, sd, potential, potential_cm, g = _gauss(D, 11)
    theta0 = torch.rand((D, C), generator=g, device="cuda") * 4 - 2
    run = bn.sample(potential, theta0, num_warmup=300, num_samples=120, seed=4, potential_cm=potential_cm,
                    state_layout="chain_major", diag_lags=12)
    assert run.samples.shape == (120, D, C) and run.inv_mass.shape == (D, C)
    assert run.num_divergent.sum() == 0 and (run.transitions == 420).all()
    x = run.samples.double()
    ess = dg.effective_sample_size(run.samples).cpu().numpy()
    mean = x.mean(dim=(0, 2)).cpu().numpy()
    std = x.permute(1, 0, 2).reshape(D, -1).std(dim=1).cpu().numpy()
    mcse = sd[:, 0].cpu().numpy() / np.sqrt(ess)
    assert np.all(np.abs(mean - mu[:, 0].cpu().numpy()) < 5 * mcse)
    np.testing.assert_allclose(std, sd[:, 0].cpu().numpy(), rtol=0.05)
    assert dg.split_rhat(run.samples).max().item() < 1.03
    np.testing.assert_allclose(run.inv_mass.mean(dim=1).cpu().numpy(), (sd[:, 0] ** 2).cpu().numpy(), rtol=0.4)
    assert 0.6 < run.accept.mean().item() < 0.95
    ref = dg.accumulate_reference(run.samples, 12)
    for k in ("ref", "sums", "lag", "ring", "head"):
        want = ref[k].cpu().numpy()
        np.testing.assert_allclose(run.diag[k].cpu().numpy(), want, rtol=2e-5, atol=2e-6 * max(1.0, np.abs(want).max()), err_msg=k)


def test_chain_major_and_chain_minor_state_take_the_same_first_transitions():
    """Same seeds, same per-chain random streams: with a fixed step size the first draws of the two layouts agree to
    rounding for (nearly) every chain -- the two kernels differ only in the order of the sums over parameters."""
    import torch

    D, C = 300, 192
    mu, sd, potential, potential_cm, g = _gauss(D, 12)
    theta0 = torch.rand((D, C), generator=g, device="cuda") * 2 - 1
    runs = [bn.sample(potential, theta0.clone(), num_warmup=0, num_samples=2, seed=9, step_size=0.05, max_tree_depth=4,
                      potential_cm=potential_cm, state_layout=lay) for lay in ("chain_minor", "chain_major")]
    a, b = runs[0].samples[0], runs[1].samples[0]  # [D, C]
    same = ((a - b).abs().max(dim=0).values < 1e-3).float().mean().item()
    assert same > 0.95, same
    close = (a - b).abs().max(dim=0).values < 1e-3  # the chains whose draws agree have the same log-density there
    assert torch.allclose(runs[0].lp[0][close], runs[1].lp[0][close], rtol=1e-3, atol=1e-2)
    assert (runs[0].num_leapfrog == runs[1].num_leapfrog).mean() > 0.9


def test_chain_major_state_on_the_wc_model():
    """NeutralWC at a size where 'auto' picks the chain-major state and the log-density call goes through its transposing
    route (C x D >= 2^22): a short run ends with every chain done, finite draws, acceptance in range."""
    import torch
    from bpl_next_b200 import Problem
    from oracle import datasets
    from tests import helpers as H

    arr = H.from_training_data("neutral_wc", datasets.config_3(), epsilon=0.1)
    p = Problem(arr)
    C = 3200
    assert C * p.D >= (1 << 22)
    g = torch.Generator(device="cuda").manual_seed(2)
    theta0 = torch.rand((p.D, C), generator=g, device="cuda") * 0.2 - 0.1

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    def potential_cm(theta, lp, grad):
        p.logdensity(theta, chain_minor=False, lp=lp, grad=grad)

    run = bn.sample(potential, theta0, num_warmup=20, num_samples=6, seed=5, max_tree_depth=4, potential_cm=potential_cm)
    assert (run.transitions == 26).all()
    assert torch.isfinite(run.samples).all() and torch.isfinite(run.lp).all()
    assert 0.3 < run.accept.mean().item() <= 1.0
    p.close()
