"""The reference's predictor classes on top of the CUDA path: same names, ``fit`` / ``predict_*`` signatures and
fitted attribute names as ``bpl/dixon_coles.py``, ``bpl/extended_dixon_coles.py``, ``bpl/neutral_dixon_coles.py`` and
``bpl/neutral_dixon_coles_WC.py`` (+ ``bpl/base.py``), so the reference's tests read the same against this package.

``fit`` = host prep (``data.prepare``) -> ``Problem`` (K1) -> batched GPU NUTS (``nuts.sample``, standing in for
``numpyro.infer.NUTS`` / ``MCMC``) -> constrained samples cut by the library's site layout -> the deterministic sites the
reference records (``attack``, ``defence``, venue effects, ``rho``, ``corr_coef``).  ``predict_*`` = K3.
``mcmc_kwargs`` understands ``num_chains`` (default 1 like numpyro; use hundreds on a GPU) and ``thin``.
"""
from __future__ import annotations

from typing import Any, Dict, Iterable, Optional, Union

import hashlib
import warnings
from datetime import datetime

import numpy as np
import torch

from . import compare as bcompare
from . import data as bdata
from . import nuts as bnuts
from . import parallel
from . import season as bseason
from .problem import Problem, pointwise_loglik, psis_loo, score_grid_host
from .problem import simulate_table as _simulate_table
from .problem import simulate_tournament as _simulate_tournament

MAX_GOALS = bdata.MAX_GOALS
# device memory for the [matches, draws] log-likelihood matrix of loo(): larger match sets are processed in ranges
LOO_MATRIX_BYTES = 4 << 30
# device memory for the raw outputs of simulate_table / simulate_tournament(return_simulations=True) (positions, scores,
# knockout entrants, scores and winners): larger runs are processed in ranges of posterior draws
SIM_OUTPUT_BYTES = 1 << 30


def _str_to_list(*args):
    return tuple([a] if isinstance(a, (str, int, np.integer)) else list(a) for a in args)  # bpl/_util.py:10-14


def constrain(flat: np.ndarray, layout: Dict[str, tuple]) -> Dict[str, np.ndarray]:
    """Flat unconstrained draws ``[S, D]`` -> dict of constrained sites (numpyro ``biject_to``: exp / clipped sigmoid)."""
    out = {}
    fi = np.finfo(np.float32)
    for name, (off, cnt, tr) in layout.items():
        x = flat[:, off:off + cnt].astype(np.float32)
        if tr == "exp":
            x = np.exp(x)
        elif tr == "sigmoid":
            x = np.clip(1.0 / (1.0 + np.exp(-x)), fi.tiny, 1.0 - fi.eps).astype(np.float32)
        out[name] = x[:, 0] if cnt == 1 and not name.endswith(("_decentered", "coefficients")) and name not in (
            "standardised_attack", "standardised_defence") else x
    return out


def _run_chains(p: Problem, num_chains: int, random_state: int, num_warmup: int, num_samples: int, thin: int, kw: dict,
                owner) -> tuple:
    """NUTS on ``num_chains`` chains of problem ``p``.  Under ``torch.distributed`` (one process per GPU) the chains are
    partitioned over the ranks -- no collective while sampling -- and the draws are all-gathered at the end, so every
    rank ends with the same ``[num_chains * num_keep, D]`` array (chains concatenated like ``MCMC.get_samples()``)."""
    rank, nranks = parallel.world()
    c0, cn = parallel.shard(num_chains, rank, nranks)
    if cn == 0:
        raise ValueError(f"num_chains={num_chains} is smaller than the number of ranks ({nranks})")
    g = torch.Generator(device="cuda").manual_seed(int(random_state))
    theta0 = torch.rand((p.D, num_chains), generator=g, device="cuda") * 4.0 - 2.0  # numpyro init_to_uniform(radius=2)
    theta0 = theta0[:, c0:c0 + cn].contiguous()

    def potential(theta, lp, grad):
        p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

    def potential_cm(theta, lp, grad):  # [chains, D] tensors: large models keep the sampler state chain-major
        p.logdensity(theta, chain_minor=False, lp=lp, grad=grad)

    kw.setdefault("potential_cm", potential_cm)
    run = bnuts.sample(potential, theta0, num_warmup=num_warmup, num_samples=num_samples, thin=thin,
                       seed=int(random_state), chain_offset=c0, **kw)
    owner.nuts_run = run
    K, D, C = run.samples.shape
    flat_dev = run.samples.permute(2, 0, 1).reshape(C * K, D).contiguous()
    if nranks > 1:
        import torch.distributed as dist
        sizes = [parallel.shard(num_chains, r, nranks)[1] * K for r in range(nranks)]
        parts = [torch.empty((n, D), dtype=flat_dev.dtype, device=flat_dev.device) for n in sizes]
        dist.all_gather(parts, flat_dev)  # the final sample gather (NCCL)
        flat_dev = torch.cat(parts, dim=0)
    _, _, cc = p.logdensity(flat_dev)  # the deterministic site "corr_coef" of every draw
    torch.cuda.synchronize()
    return flat_dev, cc


class _BplxPredictor:
    model = ""

    def __init__(self):
        self.teams = None
        self._teams_dict = None
        self.problem: Optional[Problem] = None
        self.nuts_run = None

    # ---- fit ----------------------------------------------------------------------------------------------
    def _fit(self, training_data, random_state, num_warmup, num_samples, mcmc_kwargs, epsilon=None,
             rescale_weights=False):
        kw = dict(mcmc_kwargs or {})
        num_chains = int(kw.pop("num_chains", 1))
        thin = int(kw.pop("thin", kw.pop("thinning", 1)))
        kw.pop("chain_method", None)
        kw.pop("progress_bar", None)
        arr, meta = bdata.prepare(self.model, training_data, epsilon=epsilon, rescale_weights=rescale_weights)
        self.teams, self._teams_dict = meta["teams"], meta["teams_dict"]
        self._meta = meta
        self.problem = p = Problem(arr)
        self._train_arrays = arr  # the matches log_likelihood() / waic() / loo() evaluate by default
        flat_dev, cc = _run_chains(p, num_chains, random_state, num_warmup, num_samples, thin, kw, self)
        s = constrain(flat_dev.cpu().numpy(), p.layout)
        s["corr_coef"] = cc.cpu().numpy()
        return arr, s

    def fit_streaming(self, training_data, epsilon=None, rescale_weights: bool = False, random_state: int = 42,
                      num_warmup: int = 500, num_samples: int = 1000, num_chains: int = 1024, thin: int = 10,
                      diag_lags: int = 24, max_tree_depth: int = 10, max_launches: Optional[int] = None,
                      set_posterior: bool = False, state_layout: str = "auto") -> Dict[str, Any]:
        """Many-chain ``fit`` that never stores all draws: the chains are partitioned over the ``torch.distributed`` ranks
        (no collective while sampling); every chain keeps streaming moment / lagged-product accumulators in the step
        kernel and only every ``thin``-th draw is stored.  At the end the R-hat / ESS moments are all-reduced
        (``diagnostics.streaming_summary``) and the per-chain sampler summaries all-gathered; with ``set_posterior`` the
        thinned draws are gathered too and become the fitted attributes (the ``[S, T]`` layout of
        ``neutral_dixon_coles_WC.py:308-334``), so ``predict_*`` works as after ``fit``.  Returns the run summary."""
        import time as _time

        from . import diagnostics as dg

        if self.model == "dixon_coles":
            arr, meta = bdata.prepare(self.model, training_data)
        else:
            arr, meta = bdata.prepare(self.model, training_data, epsilon=epsilon, rescale_weights=rescale_weights)
        self.teams, self._teams_dict, self._meta = meta["teams"], meta["teams_dict"], meta
        self.problem = p = Problem(arr)
        rank, nranks = parallel.world()
        c0, cn = parallel.shard(num_chains, rank, nranks)
        if cn == 0:
            raise ValueError(f"num_chains={num_chains} is smaller than the number of ranks ({nranks})")
        # numpyro init_to_uniform(radius=2), a pure function of (seed, global chain index range)
        g = torch.Generator(device="cuda").manual_seed(int(random_state) + 7919 * rank)
        theta0 = (torch.rand((p.D, cn), generator=g, device="cuda") * 4.0 - 2.0).contiguous()

        def potential(theta, lp, grad):
            p.logdensity(theta, chain_minor=True, lp=lp, grad=grad)

        def potential_cm(theta, lp, grad):  # [chains, D] tensors: large models keep the sampler state chain-major
            p.logdensity(theta, chain_minor=False, lp=lp, grad=grad)

        torch.cuda.synchronize()
        t0 = _time.perf_counter()
        run = bnuts.sample(potential, theta0, num_warmup=num_warmup, num_samples=num_samples, thin=thin,
                           seed=int(random_state), chain_offset=c0, max_tree_depth=max_tree_depth,
                           max_launches=max_launches, diag_lags=diag_lags, potential_cm=potential_cm,
                           state_layout=state_layout)
        torch.cuda.synchronize()
        t_sample = _time.perf_counter() - t0
        self.nuts_run = run
        complete_local = bool((run.transitions >= num_warmup + num_samples).all())
        # ---- the exchange: diagnostics moments (all-reduce), per-chain sampler summaries (all-gather) ---------------
        t0 = _time.perf_counter()
        summ = dg.streaming_summary(run.diag)
        per_chain = torch.from_numpy(np.stack([run.step_size, run.num_divergent.astype(np.float32),
                                               run.num_leapfrog.astype(np.float32),
                                               run.transitions.astype(np.float32)], axis=1).astype(np.float32)).cuda()
        if nranks > 1:
            import torch.distributed as dist
            parts = [torch.empty((parallel.shard(num_chains, r, nranks)[1], 4), dtype=torch.float32, device="cuda")
                     for r in range(nranks)]
            dist.all_gather(parts, per_chain)
            per_chain = torch.cat(parts, dim=0)
            launches = torch.tensor([float(run.launches)], device="cuda")
            dist.all_reduce(launches, op=dist.ReduceOp.MAX)
            launches = int(launches.item())
        else:
            launches = int(run.launches)
        torch.cuda.synchronize()
        t_exchange = _time.perf_counter() - t0
        pc = per_chain.cpu().numpy()
        complete = bool((pc[:, 3] >= num_warmup + num_samples).all())
        self.posterior_mean, self.posterior_sd = summ["mean"].cpu().numpy(), summ["sd"].cpu().numpy()
        self.rhat, self.ess = summ.get("rhat"), summ["ess"]
        out = {"complete": complete, "chains": int(pc.shape[0]), "draws_per_chain": num_samples, "thin": thin,
               "stored_draws_per_chain": int(run.samples.shape[0]), "diag_lags": int(summ["lags"]),
               "ess_min": float(summ["ess"].min().item()) if complete else 0.0,
               "ess_median": float(summ["ess"].median().item()) if complete else 0.0,
               "rhat_max": float(summ["rhat"].max().item()) if complete and "rhat" in summ else None,
               "lag_window_hit": int(summ["lag_window_hit"]),
               "leapfrogs_total": float(pc[:, 2].sum()), "leapfrogs_max_chain": float(pc[:, 2].max()),
               "logdensity_launches": launches, "divergences": int(pc[:, 1].sum()),
               "step_size_median": float(np.median(pc[:, 0])),
               "match_evals_total": float(pc[:, 2].sum()) * arr.num_matches,
               "sampling_s": t_sample, "exchange_s": t_exchange,
               "exchange": "all_reduce of (lags + 8) x D moment sums, all_gather of [chains, 4] sampler summaries"
                           + (", all_gather of the thinned draws" if set_posterior else "")}
        if set_posterior:
            K, D, C = run.samples.shape
            flat_dev = run.samples.permute(2, 0, 1).reshape(C * K, D).contiguous()
            if nranks > 1:
                import torch.distributed as dist
                sizes = [parallel.shard(num_chains, r, nranks)[1] * K for r in range(nranks)]
                parts = [torch.empty((n, D), dtype=flat_dev.dtype, device=flat_dev.device) for n in sizes]
                dist.all_gather(parts, flat_dev)
                flat_dev = torch.cat(parts, dim=0)
            _, _, cc = p.logdensity(flat_dev)
            torch.cuda.synchronize()
            s = constrain(flat_dev.cpu().numpy(), p.layout)
            s["corr_coef"] = cc.cpu().numpy()
            self._set_posterior(arr, s)
            self._train_arrays = arr
        return out

    @staticmethod
    def _prior_means(arr, s):
        S = len(s["mean_defence"])
        if arr.covariates is not None:  # extended_dixon_coles.py:138-143
            Xs = arr.covariates.astype(np.float32)
            return s["attack_coefficients"] @ Xs.T, s["mean_defence"][:, None] + s["defence_coefficients"] @ Xs.T
        return np.zeros((S, 1), np.float32), s["mean_defence"][:, None]

    # ---- predict (bpl/base.py:62-348) -------------------------------------------------------------------------
    def _parse_fixture_args(self, home_team, away_team):
        home_team, away_team = _str_to_list(home_team, away_team)
        if isinstance(home_team[0], str):
            home_team = [self._teams_dict[t] for t in home_team]
        if isinstance(away_team[0], str):
            away_team = [self._teams_dict[t] for t in away_team]
        return np.asarray(home_team, dtype=np.uint16), np.asarray(away_team, dtype=np.uint16)

    def _samples(self) -> Dict[str, np.ndarray]:
        raise NotImplementedError

    def _fixture_extras(self, n, **kw) -> Dict[str, np.ndarray]:
        return {}

    def _fixture_arrays(self, home_team, away_team, fixtures) -> Dict[str, np.ndarray]:
        """Index arrays of fixtures, mapped as ``predict_*`` maps them; the model's ``neutral_venue`` / ``home_conf`` /
        ``away_conf`` come from ``fixtures``."""
        h, a = self._parse_fixture_args(home_team, away_team)
        kw = {k: fixtures[k] for k in ("neutral_venue", "home_conf", "away_conf") if k in fixtures}
        return {"home_team": h, "away_team": a, **self._fixture_extras(len(h), **kw)}

    def _device_samples(self) -> Dict[str, torch.Tensor]:
        """The posterior draws as float32 device tensors."""
        return {k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).cuda() for k, v in self._samples().items()
                if v is not None}

    def _grid(self, home_team, away_team, max_goals, **kw):
        h, a = self._parse_fixture_args(home_team, away_team)
        fx = {"home_team": h, "away_team": a, **self._fixture_extras(len(h), **kw)}
        grid, outcome = score_grid_host(self.model, self._samples(), fx, max_goals)
        return grid, outcome

    def predict_score_grid_proba(self, home_team, away_team, *args, max_goals: int = MAX_GOALS, **kw):
        grid, _ = self._grid(home_team, away_team, max_goals, **self._extras_from_args(args, kw))
        n = np.arange(0, max_goals + 1)
        hg, ag = np.meshgrid(n, n, indexing="ij")
        return grid, hg, ag

    def predict_outcome_proba(self, home_team, away_team, *args, max_goals: int = MAX_GOALS, knockout: bool = False, **kw):
        _, out = self._grid(home_team, away_team, max_goals, **self._extras_from_args(args, kw))
        hw, dr, aw = out[:, 0], out[:, 1], out[:, 2]
        if knockout:  # neutral_dixon_coles.py:650-653
            norm = hw + aw
            return {"home_win": hw / norm, "away_win": aw / norm}
        return {"home_win": hw, "draw": dr, "away_win": aw}

    def predict_score_proba(self, home_team, away_team, home_goals, away_goals, *args, **kw):
        home_goals, away_goals = _str_to_list(home_goals, away_goals)
        hg, ag = np.asarray(home_goals, dtype=np.int64), np.asarray(away_goals, dtype=np.int64)
        mg = int(max(hg.max(), ag.max(), 1))
        grid, _ = self._grid(home_team, away_team, mg, **self._extras_from_args(args, kw))
        if len(hg) == 1 and grid.shape[0] > 1:
            hg, ag = np.repeat(hg, grid.shape[0]), np.repeat(ag, grid.shape[0])
        return grid[np.arange(grid.shape[0]), hg, ag]

    def _n_proba(self, n, team, opponent, home, max_goals, scored, **kw):
        n = [n] if isinstance(n, (int, np.integer)) else list(np.asarray(n))
        grid, _ = self._grid(team, opponent, max_goals, **kw) if home else self._grid(opponent, team, max_goals, **kw)
        # marginal of the grid: sum over the other side's goals (bpl/base.py:248-348)
        team_axis_is_home = home if scored else not home
        marg = grid.sum(axis=2) if team_axis_is_home else grid.sum(axis=1)  # [F, g]
        return marg[0, np.asarray(n, dtype=np.int64)]

    def predict_score_n_proba(self, n, team, opponent, home: bool = True, max_goals: int = MAX_GOALS, **kw):
        return self._n_proba(n, team, opponent, home, max_goals, True, **kw)

    def predict_concede_n_proba(self, n, team, opponent, home: bool = True, max_goals: int = MAX_GOALS, **kw):
        return self._n_proba(n, team, opponent, home, max_goals, False, **kw)

    def _extras_from_args(self, args, kw):
        return kw

    # ---- model comparison: pointwise log-likelihood, WAIC, PSIS-LOO, held-out log score ------------------------
    # ll[s, m] = log Pois(yh; lh) + log Pois(ya; la) + log tau(yh, ya; lh, la, corr_coef_s), with the rates of the predict
    # path (neutral venues, confederations; Extended's fit-time clip of the rates at 15 is not applied), tau clamped at 0
    # (a match can give -inf) and NO match weights: exp(ll) averaged over s is what predict_score_proba returns.
    def _observations(self, data=None):
        """Observed matches as index / goal arrays (the training data when ``data`` is None), and a key naming them."""
        if data is None:
            arr = getattr(self, "_train_arrays", None)
            if arr is None:
                raise ValueError("no training data recorded: fit the model first, or pass data")
            obs = {"home_team": arr.home_team, "away_team": arr.away_team}
            for k in ("neutral_venue", "home_conf", "away_conf"):
                if getattr(arr, k) is not None:
                    obs[k] = np.asarray(getattr(arr, k), dtype=np.uint8)
            hg, ag = arr.home_goals, arr.away_goals
        else:
            obs = self._fixture_arrays(data["home_team"], data["away_team"], data)
            hg, ag = bdata._goals(data["home_goals"]), bdata._goals(data["away_goals"])
        obs["home_goals"], obs["away_goals"] = np.asarray(hg, dtype=np.uint8), np.asarray(ag, dtype=np.uint8)
        names = np.asarray(self.teams).astype(str)
        key = hashlib.sha1("|".join(names[obs["home_team"].astype(np.int64)]).encode())
        key.update("|".join(names[obs["away_team"].astype(np.int64)]).encode())
        key.update(obs["home_goals"].tobytes() + obs["away_goals"].tobytes())
        return obs, key.hexdigest()

    def _comparison_inputs(self, data):
        obs, key = self._observations(data)
        ds = self._device_samples()
        do = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in obs.items()}
        return ds, do, key

    def log_likelihood(self, data=None) -> np.ndarray:
        """Pointwise log-likelihood ``[S, M]`` float32 (numpyro's ``log_likelihood`` shape: draws x observations) of
        the observed scores of ``data`` (reference ``training_data`` keys; default: the training data).

        ``ll[s, m] = log Pois(yh; lh) + log Pois(ya; la) + log tau(yh, ya; lh, la, corr_coef_s)``: the rates are those of
        ``predict_*`` (neutral venues and confederations included; Extended's fit-time clip of rates at 15 is not
        applied), tau is clamped at 0 so a match can give -inf, and the value is UNWEIGHTED -- for a fit with time decay
        or game weights it is the predictive density of the match, not the weighted pseudo-likelihood that was fitted.
        ``exp(ll)`` averaged over the draws is what ``predict_score_proba`` returns for that match."""
        ds, do, _ = self._comparison_inputs(data)
        ll, _ = pointwise_loglik(self.model, ds, do)
        return np.ascontiguousarray(ll.cpu().numpy().T)

    def waic(self, data=None) -> Dict[str, Any]:
        """WAIC of the fit on ``data`` (default: the training data), from the pointwise log-likelihood of
        ``log_likelihood`` (unweighted; see there) without storing it:
        ``lppd_m = logsumexp_s ll - log S``, ``p_waic_m = var_s ll`` with divisor S (ddof 0),
        ``elpd_waic_m = lppd_m - p_waic_m``.  Returns ``elpd_waic`` (sum), ``se = sqrt(M var0(elpd_waic_m))``,
        ``p_waic``, ``lppd``, the pointwise arrays and ``match_key`` (names the matches, for ``compare``)."""
        ds, do, key = self._comparison_inputs(data)
        _, st = pointwise_loglik(self.model, ds, do, want_matrix=False)
        return bcompare.waic_from_stats(st.cpu().numpy(), int(ds["attack"].shape[0]), key)

    def loo(self, r_eff: float = 1.0) -> Dict[str, Any]:
        """Pareto-smoothed importance-sampling leave-one-out cross-validation on the training data (ArviZ's ``loo``;
        Vehtari et al., JMLR 2024), every step on the GPU.  Per match m the log-ratios ``-ll[:, m]`` of
        ``log_likelihood`` (unweighted: for a fit with time decay or game weights this evaluates predictive density, not
        the weighted pseudo-likelihood that was fitted) get a generalised-Pareto-smoothed tail of
        ``ceil(min(0.2 S, 3 sqrt(S / r_eff)))`` draws, and ``elpd_loo_m = logsumexp_s(lw + ll)``.

        Returns ``elpd_loo = sum_m elpd_loo_m``, ``se = sqrt(M var0(elpd_loo_m))``, ``p_loo = sum_m lppd_m - elpd_loo``,
        ``pointwise`` (``elpd_loo_m``), ``pareto_k`` (k-hat per match; +inf when the tail has at most 4 draws),
        ``good_k = min(1 - 1/log10 S, 0.7)`` with ``n_k_above_good`` and ``n_k_above_0.7`` (the counts of unreliable
        matches), ``r_eff`` (one scalar relative efficiency for every match) and ``match_key``.  A match whose
        log-likelihood is not finite in some draw gets ``elpd_loo_m`` NaN and k-hat +inf.  The ``[M, S]`` matrix is
        computed and smoothed in ranges of matches that keep it within ``LOO_MATRIX_BYTES`` of device memory; the
        results do not depend on the range size.  To choose ``epsilon`` (time decay) use ``log_score`` on later
        matches instead."""
        import torch

        ds, do, key = self._comparison_inputs(None)
        S, M = int(ds["attack"].shape[0]), int(do["home_team"].shape[0])
        rows = max(1, min(M, LOO_MATRIX_BYTES // (4 * S)))
        buf = torch.empty((rows, S), dtype=torch.float32, device="cuda")
        elpd, khat, lppd = [], [], []
        for lo in range(0, M, rows):
            hi = min(M, lo + rows)
            ll, st = pointwise_loglik(self.model, ds, {k: v[lo:hi] for k, v in do.items()}, loglik=buf)
            e, k = psis_loo(ll, r_eff)
            elpd.append(e.cpu().numpy())
            khat.append(k.cpu().numpy())
            lppd.append(bcompare.lppd_from_stats(st.cpu().numpy(), S))
        return bcompare.loo_from_pointwise(np.concatenate(elpd), np.concatenate(khat), np.concatenate(lppd), S, r_eff,
                                           key)

    def log_score(self, data) -> Dict[str, Any]:
        """Held-out log score of the posterior predictive on ``data`` (matches not used in the fit, reference
        ``training_data`` keys): ``log_score = sum_m lppd_m`` with ``lppd_m = log((1/S) sum_s exp(ll[s, m]))``, the log
        of the probability ``predict_score_proba`` gives the observed score (``pointwise``).  The way to choose
        ``epsilon`` / ``rescale_weights``: fit on earlier matches, score later ones."""
        ds, do, _ = self._comparison_inputs(data)
        _, st = pointwise_loglik(self.model, ds, do, want_matrix=False)
        lppd = bcompare.lppd_from_stats(st.cpu().numpy(), int(ds["attack"].shape[0]))
        return {"log_score": float(lppd.sum()), "pointwise": lppd, "num_matches": len(lppd)}

    # ---- posterior predictive checks ------------------------------------------------------------------------------
    def posterior_predictive_check(self, data=None, num_sims_per_draw: int = 1, random_state: Optional[int] = None,
                                   max_goals: int = MAX_GOALS, score_bins: int = 6, points=(3, 1),
                                   return_replicates: bool = False) -> Dict[str, Any]:
        """Does the fit reproduce the data? Replicated datasets of the observed matches of ``data`` (reference
        ``training_data`` keys; default: the training data) are drawn on the GPU, one posterior draw per replicate, and
        their statistics are set beside those of the observed scores.

        Replicate ``n = (first_draw + s) R + r`` (R = ``num_sims_per_draw``) uses draw s; every match of it is drawn by
        ``simulate_table``'s sampler (the draw's own grid up to ``max_goals``, tau clamped at 0, normalised by its sum;
        the rates of ``predict_*``), from Philox words 2m and 2m + 1 of ``curand_init(seed, n, 0)``, so with the same
        seed and matches the replicated scores are ``simulate_table``'s.  Match weights are ignored: for a time-decayed
        fit every match counts equally; pass ``data`` (the last season, say) to check recent form.

        Statistics: ``score_counts [B, B]`` (matches per cell ``min(hg, B-1), min(ag, B-1)``, B = ``score_bins``: with 6,
        0-4 and "5+"), ``outcome_counts [3]`` (home wins, draws, away wins), ``goals [2]`` (home, away),
        ``total_goals_sq`` (sum of squared match totals), ``total_goals_dispersion`` (variance over mean of total goals
        per match: 1 for Poisson totals), and per team ``team_points`` (``points`` = (win, draw)), ``team_goals_for``,
        ``team_goals_against [T]`` in the order of ``teams``.  Each maps to ``observed``, ``mean`` and ``sd`` over the
        N = S R replicates and ``p_value``, the mid-p ``P(T_rep > T_obs) + 1/2 P(T_rep = T_obs)``: near 0.5 the data
        sit inside what the model predicts, near 0 or 1 the model misses (a team with no matches gets 0.5).  Observed
        goals above ``max_goals`` count as they are; replicated goals cannot exceed it.

        Also returned: ``teams``, ``score_bins``, ``max_goals``, ``num_replicates``, ``sims_per_draw``, ``seed`` (from
        the clock when ``random_state`` is None; pass it back to repeat the run) and ``match_key`` (names the matches).
        With ``return_replicates``, ``replicates`` (each statistic per replicate, ``[N, ...]``) and ``home_score`` /
        ``away_score [M, N]`` (``sample_score``'s shape).  The draws run in ranges within ``SIM_OUTPUT_BYTES`` of device
        output; the results do not depend on the range size.  Raises if a replicate met a non-finite rate."""
        if self.teams is None:
            raise ValueError("the model is not fitted: fit it first")
        from . import ppc as bppc
        from .problem import posterior_predictive

        seed = int(datetime.now().timestamp() * 100) if random_state is None else int(random_state)
        R, B = int(num_sims_per_draw), int(score_bins)
        if R < 1:
            raise ValueError(f"num_sims_per_draw must be >= 1, got {num_sims_per_draw}")
        ds, do, key = self._comparison_inputs(data)
        S, T, M = int(ds["attack"].shape[0]), int(ds["attack"].shape[1]), int(do["home_team"].shape[0])
        step = (2 ** 31 - 1) // R  # replicates per call stay below 2^31
        per_rep = 4 * (B * B + 3 + 3 * T) + 8 * 3 + (2 * M if return_replicates else 0)  # device output bytes
        step = min(step, max(1, SIM_OUTPUT_BYTES // (R * per_rep)))
        parts, scores, invalid = [], [], 0
        for lo in range(0, S, step):
            hi = min(S, lo + step)
            out = posterior_predictive(self.model, {k: v[lo:hi] for k, v in ds.items()}, do, max_goals, B, points, R,
                                       seed, first_draw=lo, want_scores=return_replicates)
            invalid += int(out["invalid"].item())
            parts.append({k: out[k].cpu().numpy() for k in bppc.STATISTICS})
            if return_replicates:
                scores.append(out["scores"].cpu().numpy())
        N = S * R
        if invalid:
            raise ValueError(f"{invalid} of {N} replicates met a non-finite scoring rate or score-grid normaliser: "
                             "check the posterior draws")
        reps = {k: np.concatenate([p[k] for p in parts]) for k in bppc.STATISTICS}
        h = {k: do[k].cpu().numpy() for k in ("home_team", "away_team", "home_goals", "away_goals")}
        observed = bppc.statistics(h["home_team"], h["away_team"], h["home_goals"], h["away_goals"], T, B, points)
        res = bppc.summarize(observed, reps, M)
        res.update(teams=list(np.asarray(self.teams).tolist()), score_bins=B, max_goals=int(max_goals),
                   num_replicates=N, sims_per_draw=R, seed=seed, match_key=key)
        if return_replicates:
            sc = np.concatenate(scores)
            res.update(replicates=reps, home_score=np.ascontiguousarray(sc[:, :, 0].T),
                       away_score=np.ascontiguousarray(sc[:, :, 1].T))
        return res

    # ---- simulation from the grid (bpl/base.py:150-246, bpl/_util.py:96-112) -----------------------------------
    @staticmethod
    def _choice(probs: np.ndarray, num_samples: int, random_state) -> np.ndarray:
        """``[F, K]`` probabilities -> ``[F, num_samples]`` category indices, one independent stream per fixture (the
        reference draws with ``jax.random.choice`` under ``vmap``; like it, the row is normalised by its own sum)."""
        if random_state is None:
            random_state = int(datetime.now().timestamp() * 100)
        rng = np.random.default_rng(int(random_state))
        cdf = np.cumsum(probs.astype(np.float64), axis=1)
        u = rng.random((probs.shape[0], int(num_samples))) * cdf[:, -1:]
        idx = (u[:, :, None] >= cdf[:, None, :]).sum(axis=2)
        return np.minimum(idx, probs.shape[1] - 1)

    def _sample_score(self, home_team, away_team, num_samples, random_state, max_goals, **kw):
        grid, hg, ag = _BplxPredictor.predict_score_grid_proba(self, home_team, away_team, max_goals=max_goals, **kw)
        idx = self._choice(grid.reshape(grid.shape[0], -1), num_samples, random_state)
        return {"home_score": hg.ravel()[idx], "away_score": ag.ravel()[idx]}

    def _sample_outcome(self, home_team, away_team, num_samples, random_state, max_goals, knockout=False, **kw):
        h, a = self._parse_fixture_args(home_team, away_team)
        pr = _BplxPredictor.predict_outcome_proba(self, h, a, max_goals=max_goals, knockout=knockout, **kw)
        keys = ("home_win", "away_win") if knockout else ("home_win", "draw", "away_win")
        idx = self._choice(np.stack([pr[k] for k in keys], axis=1), num_samples, random_state)
        names = np.append(np.asarray(self.teams), "Draw")
        draw = len(self.teams)
        hrep, arep = np.repeat(h[:, None], num_samples, axis=1).astype(np.int64), np.repeat(a[:, None], num_samples, axis=1).astype(np.int64)
        away_code = 1 if knockout else 2
        winner = np.where(idx == 0, hrep, np.where(idx == away_code, arep, draw))
        return names[winner]

    def sample_score(self, home_team, away_team, num_samples: int = 1, random_state: Optional[int] = None,
                     max_goals: int = MAX_GOALS):
        """``{"home_score", "away_score"}``, each ``[fixtures, num_samples]`` (``bpl/base.py:150-195``)."""
        return self._sample_score(home_team, away_team, num_samples, random_state, max_goals)

    def sample_outcome(self, home_team, away_team, num_samples: int = 1, random_state: Optional[int] = None,
                       max_goals: int = MAX_GOALS):
        """``[fixtures, num_samples]`` names of the winning team, or ``"Draw"`` (``bpl/base.py:197-246``)."""
        return self._sample_outcome(home_team, away_team, num_samples, random_state, max_goals)

    # ---- season / group-stage simulation -------------------------------------------------------------------------
    def simulate_table(self, fixtures, played=None, teams=None, groups=None, num_sims_per_draw: int = 1,
                       random_state: Optional[int] = None, max_goals: int = MAX_GOALS, points=(3, 1),
                       return_simulations: bool = False, tiebreak: str = "goal_difference") -> Dict[str, Any]:
        """Finishing-position and points probabilities of a league table or of group tables, simulated on the GPU.

        Every simulated season takes ONE posterior draw and plays every remaining fixture with that draw's rates, so a
        team that is stronger in a draw is stronger in all of its matches of that season (sampling fixtures one by one,
        as ``sample_score`` does, loses that correlation and makes the spread of final points too narrow).  Each of the
        S draws gives ``num_sims_per_draw`` seasons: ``num_simulations = S * num_sims_per_draw``.

        ``fixtures``: the remaining matches with reference ``training_data`` keys (``home_team``, ``away_team``, and
        ``neutral_venue`` / ``home_conf`` / ``away_conf`` where the model has them, mapped as ``predict_*`` maps them).
        ``played``: results so far (``home_team``, ``away_team``, ``home_goals``, ``away_goals``) that make the starting
        table.  ``teams``: the table (default: the sorted union of the teams in ``fixtures`` and ``played``); every team
        in a fixture must be known to the model and in the table, and at most 64 teams are supported.  ``groups``: a
        mapping team -> group label, or labels aligned with ``teams``; teams are then ranked within their group.
        ``points``: (win, draw).

        A fixture's score is drawn from the draw's own score grid up to ``max_goals`` (tau clamped at 0, normalised by
        its sum); averaged over draws this is ``predict_score_grid_proba``.  ``tiebreak`` says how teams level on
        points are ranked within their group:

        * ``"goal_difference"`` (default): goal difference, goals for, then a random key.
        * ``"head_to_head"`` (UEFA group stages, La Liga, Serie A): for a set of teams level on points, the points, goal
          difference and goals for of the matches among them only (in ``played`` and the simulated ``fixtures``);
          teams still level on all three go through that again with only the matches among themselves; a set it does
          not separate at all (teams that have not met, say) is ordered by overall goal difference, goals for, then
          the random key.

        Fair-play rules are NOT modelled: ties left at the end are decided by lot.  Both rules read the same random
        numbers, so with the same seed they differ only in the order of teams level on points.

        Returns ``teams``, ``groups`` (each team's label, or None), ``tiebreak`` (the rule that ranked the table),
        ``position_proba [T, P]`` (P = the largest group;
        position 0 = first), ``points_proba [T, B]`` (points GAINED in ``fixtures``), ``start_points``,
        ``expected_points`` (final), ``num_simulations``, ``sims_per_draw`` and ``seed`` (from the clock when
        ``random_state`` is None; pass it back to repeat the run).  With ``return_simulations`` also ``positions [N, T]``
        and ``home_score`` / ``away_score`` ``[F, N]`` (``sample_score``'s shape); the draws are then processed in
        ranges that keep these within ``SIM_OUTPUT_BYTES`` of device memory, and the results do not depend on the range
        size.  Raises if any simulation met a non-finite rate."""
        home, away = _str_to_list(fixtures["home_team"], fixtures["away_team"])
        tteams = bseason.table_teams(home, away, played, teams)
        table = bseason.build_table(tteams, played, groups, points, tiebreak)
        hs, as_ = bseason.fixture_slots(table, home, away, known_teams=self.teams)
        fx = {**self._fixture_arrays(home, away, fixtures), "home_slot": hs, "away_slot": as_}
        return self._simulate(table, fx, None, num_sims_per_draw, random_state, max_goals, return_simulations,
                              "met a non-finite scoring rate or score-grid normaliser: check the posterior draws")

    def _simulate(self, table, fx, bracket, num_sims_per_draw, random_state, max_goals, return_simulations,
                  invalid_reason) -> Dict[str, Any]:
        """``simulate_table`` (``bracket`` None) and ``simulate_tournament`` from the host table, fixture arrays (with
        their slots; ``{}`` for none) and bracket: the draws in ranges, counts summed over the ranges, probabilities."""
        seed = int(datetime.now().timestamp() * 100) if random_state is None else int(random_state)
        R = int(num_sims_per_draw)
        if R < 1:
            raise ValueError(f"num_sims_per_draw must be >= 1, got {num_sims_per_draw}")
        ds = self._device_samples()
        dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fx.items()}
        dtab = {k: None if table[k] is None else torch.from_numpy(table[k]).cuda()
                for k in ("start_points", "start_goals_for", "start_goals_against", "group")}
        dtab.update({k: table[k] for k in ("num_positions", "num_points_bins", "points_win", "points_draw")})
        dtab.update(tiebreak=table.get("tiebreak", "goal_difference"), played_h2h=table.get("played_h2h"))  # (host)
        S, T, F = int(ds["attack"].shape[0]), len(table["teams"]), len(fx.get("home_team", ()))
        K = 0 if bracket is None else len(bracket["round"])
        step = (2 ** 31 - 1) // R  # simulations per call stay below 2^31
        if return_simulations:  # bytes per simulation: positions, scores, the knockout entrants, scores, winners, extra
            step = min(step, max(1, SIM_OUTPUT_BYTES // (R * (T + 2 * F + 9 * K))))
        if step < 1:
            raise ValueError(f"num_sims_per_draw={R} is too large for one draw per call")
        acc, invalid, raw = {}, 0, []
        for lo in range(0, S, step):
            hi = min(S, lo + step)
            draws = {k: v[lo:hi] for k, v in ds.items()}
            if bracket is None:
                out = _simulate_table(self.model, draws, dfx, dtab, max_goals, R, seed, first_draw=lo,
                                      want_positions=return_simulations, want_scores=return_simulations)
            else:
                out = _simulate_tournament(self.model, draws, dfx, dtab, bracket, max_goals, R, seed, first_draw=lo,
                                           want_positions=return_simulations, want_scores=return_simulations,
                                           want_knockout=return_simulations)
            invalid += int(out.pop("invalid").item())
            for k, v in out.items():
                if k.endswith("_counts"):
                    acc[k] = v if k not in acc else acc[k] + v
            if return_simulations:
                raw.append({k: v.cpu().numpy() for k, v in out.items() if not k.endswith("_counts")})
        N = S * R
        if invalid:
            raise ValueError(f"{invalid} of {N} simulations {invalid_reason}")
        cnt = {k: v.cpu().numpy() for k, v in acc.items()}
        res = {"teams": table["teams"],
               "groups": None if table["group"] is None else [table["group_labels"][g] for g in table["group"]],
               "tiebreak": dtab["tiebreak"],
               **bseason.probabilities(table, cnt["position_counts"], cnt["points_counts"], N)}
        if bracket is not None:
            res.update(bseason.bracket_probabilities(bracket, cnt["reach_counts"], cnt["win_counts"], N,
                                                     cnt["decided_counts"]))
        res.update({"start_points": table["start_points"].astype(np.int64), "num_simulations": N, "sims_per_draw": R,
                    "seed": seed})
        if return_simulations:
            cat = {k: np.concatenate([r[k] for r in raw]) for k in raw[0]}
            sc = cat.pop("scores")
            res.update(positions=cat.pop("positions"), home_score=np.ascontiguousarray(sc[:, :, 0].T),
                       away_score=np.ascontiguousarray(sc[:, :, 1].T), **cat)
        return res

    def _slot_confs(self, tteams, fixtures, team_conf):
        """Confederation index of every table team (NeutralWC): ``team_conf`` (team -> name or index), else inferred
        from the group fixtures, which must then give each team one confederation."""
        conf = {}
        if team_conf is None and fixtures is not None and "home_conf" in fixtures:
            for side in ("home", "away"):
                for t, c in zip(_str_to_list(fixtures[side + "_team"])[0], _str_to_list(fixtures[side + "_conf"])[0]):
                    if conf.setdefault(t, c) != c:
                        raise ValueError(f"team {t!r} plays for confederations {conf[t]!r} and {c!r} in the fixtures: "
                                         "pass team_conf")
        elif team_conf is not None:
            conf = dict(team_conf)
        missing = [t for t in tteams if t not in conf]
        if missing:
            raise ValueError(f"the confederation of {missing[:3]!r} is unknown: pass team_conf")
        return np.asarray([self._conferences_dict[conf[t]] if isinstance(conf[t], str) else int(conf[t])
                           for t in tteams], np.uint8)

    def simulate_tournament(self, fixtures, bracket, played=None, teams=None, groups=None, best=None, team_conf=None,
                            num_sims_per_draw: int = 1, random_state: Optional[int] = None, max_goals: int = MAX_GOALS,
                            points=(3, 1), return_simulations: bool = False,
                            tiebreak: str = "goal_difference") -> Dict[str, Any]:
        """A tournament simulated on the GPU: the group stage of ``simulate_table``, then a knockout bracket, with ONE
        posterior draw per simulated tournament, so a team that is stronger in a draw is stronger in every match of its
        path.  (Chaining ``predict_outcome_proba`` calls cannot give this: the opponent of a round depends on earlier
        results, and the same uncertain strengths run through all of a team's matches.)

        ``fixtures``, ``played``, ``teams``, ``groups``, ``points``, ``num_sims_per_draw``, ``random_state``,
        ``max_goals``, ``tiebreak``: as ``simulate_table`` (``"head_to_head"`` ranks each group by the matches among
        its teams level on points, as UEFA's and FIFA's group stages do); ``fixtures`` may be None or empty (a cup whose draw is made: the entrants
        are ``("team", name)``).  ``bracket``: the ties in play order, ``{"id", "round", "home", "away",
        "neutral_venue", "format"}``, entrants ``("group", label, position)``, ``("best", j)``, ``("winner", id)``,
        ``("loser", id)`` or ``("team", name)``; ``best``: the best-placed qualifiers, ``{"position", "count",
        "allocation"}`` (``season.build_bracket``).  ``team_conf`` (NeutralWC): team -> confederation, needed for the
        ties; inferred from the fixtures' confederations when they are consistent.

        A tie's ``format`` is one of:

        * ``"one_match"`` (default): one match, played like a group fixture from the draw's own grid.  A drawn tie goes
          to the home entrant with probability ``hw_s / (hw_s + aw_s)``, the draw's own home and away win masses: the
          per-draw form of the knockout renormalisation, which differs from ``predict_outcome_proba(knockout=True)``
          (that renormalises after averaging over the draws).
        * ``"extra_time"``: one match; if it is drawn, extra time is played at the same venue; if that is also level,
          penalties.
        * ``"two_legs"``: ``home`` hosts leg 1 and ``away`` hosts leg 2 with the venues swapped (never at a neutral
          venue); the higher aggregate goes through (no away-goals rule); level on aggregate: extra time in leg 2, then
          penalties.

        Each leg is a 90-minute match from the draw's own grid.  Extra time uses the draw's rates times 1/3 (30 of 90
        minutes at the model's constant rates) with no tau correction; the home entrant wins a shoot-out with
        probability 1/2 (the model knows nothing of penalties).  Best-placed teams are ranked across groups by
        points, goal difference, goals for, then lot, under either ``tiebreak`` (teams of different groups have no
        head-to-head).

        Returns everything ``simulate_table`` returns, plus ``rounds`` (labels by first appearance), ``reach_proba`` /
        ``win_proba [T, rounds]`` (the team plays / wins a tie of the round; a two-legged tie counts once),
        ``champion_proba [T]``, ``tie_ids`` and ``decided_proba [K, 3]`` (tie k settled in normal time or on aggregate,
        in extra time, or by penalties / the per-draw lot).  With ``return_simulations`` also ``positions [N, T]``,
        ``home_score`` / ``away_score [F, N]``, ``ko_entrants [N, K, 2]`` (table slots), ``ko_scores [N, K, 2]`` (the
        first or only match), ``ko_winners [N, K]`` and ``ko_extra [N, K, 4]`` (leg-2 goals of home and away entrant,
        then their extra-time goals; 254 where not played); the draws are then processed in ranges
        within ``SIM_OUTPUT_BYTES`` and the results do not depend on the range size.  Raises if a simulation was invalid
        (a non-finite rate, or an allocation row the bracket does not cover)."""
        fixtures = fixtures if fixtures is not None and len(_str_to_list(fixtures["home_team"])[0]) else None
        home, away = _str_to_list(fixtures["home_team"], fixtures["away_team"]) if fixtures else ([], [])
        named = [e[1] for tie in bracket for e in (tuple(tie["home"]), tuple(tie["away"])) if e[0] == "team"]
        if teams is None:
            tteams = bseason.table_teams(home + named, away, played) if (home or named or played) else []
        else:
            tteams = bseason.table_teams(home, away, played, teams)
        table = bseason.build_table(tteams, played, groups, points, tiebreak)
        br = bseason.build_bracket(table, bracket, best)
        known = set(np.asarray(self.teams).tolist())
        unknown = [t for t in tteams if t not in known]
        if unknown:
            raise ValueError(f"team {unknown[0]!r} is not known to the model")
        br["slot_team"] = np.asarray([self._teams_dict[t] for t in tteams], np.uint16)
        if self.model == "neutral_wc":
            br["slot_conf"] = self._slot_confs(tteams, fixtures, team_conf)
        if fixtures:
            hs, as_ = bseason.fixture_slots(table, home, away, known_teams=self.teams)
            fx = {**self._fixture_arrays(home, away, fixtures), "home_slot": hs, "away_slot": as_}
        else:
            fx = {}
            bseason._size_histograms(table)
        return self._simulate(table, fx, br, num_sims_per_draw, random_state, max_goals, return_simulations,
                              "were invalid: a non-finite scoring rate or score-grid normaliser (check the posterior "
                              "draws), or best-placed qualifiers the bracket does not place")

    # ---- a team the model has not seen (extended_dixon_coles.py:401-462 and the neutral siblings) ---------------
    def _new_team_pair(self, team_name, team_covariates):
        """Draws of (attack, defence) for a new team from the fitted hierarchical prior, one per posterior sample."""
        if team_name in self.teams:
            raise ValueError(f"Team {team_name} already known to model.")
        if self.attack_coefficients is not None:
            if team_covariates is None:
                warnings.warn(f"You haven't provided features for {team_name}. Assuming team_covariates are the average of "
                              "known teams. For better forecasts, provide team_covariates.")
                x = np.zeros(self.attack_coefficients.shape[1], np.float32)
            else:
                x = (0.5 * (np.asarray(team_covariates, np.float32) - self._meta["team_covariates_mean"])
                     / self._meta["team_covariates_std"]).ravel()
            mean_attack = self.attack_coefficients @ x
            mean_defence = self.mean_defence + self.defence_coefficients @ x
        else:
            mean_attack, mean_defence = 0.0, self.mean_defence
        a_tilde = np.random.normal(loc=0.0, scale=1.0, size=len(self.std_attack))
        b_tilde = np.random.normal(loc=self.rho * a_tilde, scale=np.sqrt(1.0 - self.rho ** 2.0))
        return mean_attack + a_tilde * self.std_attack, mean_defence + b_tilde * self.std_defence

    def _append_team(self, team_name, columns: Dict[str, np.ndarray]):
        self.teams = np.append(self.teams, team_name)
        self._teams_dict[team_name] = len(self._teams_dict)
        for name, col in columns.items():
            setattr(self, name, np.concatenate((getattr(self, name), np.asarray(col, np.float32)[:, None]), axis=1))


class DixonColesMatchPredictor(_BplxPredictor):
    """``bpl/dixon_coles.py:26-163``."""
    model = "dixon_coles"

    def fit(self, training_data, random_state: int = 42, num_warmup: int = 500, num_samples: int = 1000,
            mcmc_kwargs: Optional[Dict[str, Any]] = None, run_kwargs: Optional[Dict[str, Any]] = None):
        arr, s = self._fit(training_data, random_state, num_warmup, num_samples, mcmc_kwargs)
        return self._set_posterior(arr, s)

    def _set_posterior(self, arr, s):
        """Constrained draws of the latent sites -> the sites the reference records (dixon_coles.py:52-61)."""
        self.attack = s["std_attack"][:, None] * s["attack_decentered"]
        self.defence = s["mean_defence"][:, None] + s["std_defence"][:, None] * s["defence_decentered"]
        self.home_advantage = s["home_advantage"]
        self.corr_coef = s["corr_coef"]
        return self

    def _samples(self):
        return {"attack": self.attack, "defence": self.defence, "home_advantage": self.home_advantage,
                "corr_coef": self.corr_coef}


class ExtendedDixonColesMatchPredictor(_BplxPredictor):
    """``bpl/extended_dixon_coles.py:28-462``."""
    model = "extended"

    def fit(self, training_data, random_state: int = 42, num_warmup: int = 500, num_samples: int = 1000,
            epsilon: Optional[float] = None, rescale_weights: bool = False,
            mcmc_kwargs: Optional[Dict[str, Any]] = None, run_kwargs: Optional[Dict[str, Any]] = None):
        arr, s = self._fit(training_data, random_state, num_warmup, num_samples, mcmc_kwargs, epsilon, rescale_weights)
        return self._set_posterior(arr, s)

    def _set_posterior(self, arr, s):
        """Constrained draws of the latent sites -> the sites the reference records (extended_dixon_coles.py:182-187)."""
        am, dm = self._prior_means(arr, s)
        self.attack = am + s["standardised_attack"] * s["std_attack"][:, None]
        self.defence = dm + s["standardised_defence"] * s["std_defence"][:, None]
        self.home_advantage = s["mean_home_advantage"][:, None] + s["std_home_advantage"][:, None] * s["home_advantage_decentered"]
        self.corr_coef = s["corr_coef"]
        self.u = s["u"]
        self.rho = 2.0 * s["u"] - 1.0
        self.mean_defence, self.std_attack, self.std_defence = s["mean_defence"], s["std_attack"], s["std_defence"]
        self.mean_home_advantage, self.std_home_advantage = s["mean_home_advantage"], s["std_home_advantage"]
        self.standardised_attack, self.standardised_defence = s["standardised_attack"], s["standardised_defence"]
        self.attack_coefficients = s.get("attack_coefficients") if arr.covariates is not None else None
        self.defence_coefficients = s.get("defence_coefficients") if arr.covariates is not None else None
        return self

    def _samples(self):
        return {"attack": self.attack, "defence": self.defence, "home_advantage": self.home_advantage,
                "corr_coef": self.corr_coef}

    def add_new_team(self, team_name: str, team_covariates: Optional[np.ndarray] = None) -> None:
        """Parameters for a team not seen in training, drawn from the fitted priors (``extended_dixon_coles.py:401-462``;
        like the reference this uses numpy's global random state)."""
        attack, defence = self._new_team_pair(team_name, team_covariates)
        home_advantage = np.random.normal(loc=self.mean_home_advantage, scale=self.std_home_advantage)
        self._append_team(team_name, {"attack": attack, "defence": defence, "home_advantage": home_advantage})


class NeutralDixonColesMatchPredictor(_BplxPredictor):
    """``bpl/neutral_dixon_coles.py:31-902`` (signatures as there: ``neutral_venue`` is a positional fixture argument)."""
    model = "neutral"
    _effects = ("home_attack", "away_attack", "home_defence", "away_defence")

    def fit(self, training_data, epsilon: Optional[float] = None, rescale_weights: bool = False, random_state: int = 42,
            num_warmup: int = 500, num_samples: int = 1000, mcmc_kwargs: Optional[Dict[str, Any]] = None,
            run_kwargs: Optional[Dict[str, Any]] = None):
        arr, s = self._fit(training_data, random_state, num_warmup, num_samples, mcmc_kwargs, epsilon, rescale_weights)
        return self._set_posterior(arr, s)

    def _set_posterior(self, arr, s):
        """Constrained draws of the latent sites -> the sites the reference records."""
        am, dm = self._prior_means(arr, s)
        self.attack = am + s["standardised_attack"] * s["std_attack"][:, None]
        self.defence = dm + s["standardised_defence"] * s["std_defence"][:, None]
        for nm in self._effects:  # neutral_dixon_coles.py:205-224
            setattr(self, nm, s["mean_" + nm][:, None] + s["std_" + nm][:, None] * s[nm + "_decentered"])
            setattr(self, "mean_" + nm, s["mean_" + nm])
            setattr(self, "std_" + nm, s["std_" + nm])
        self.corr_coef = s["corr_coef"]
        self.u = s["u"]
        self.rho = 2.0 * s["u"] - 1.0
        self.mean_defence, self.std_attack, self.std_defence = s["mean_defence"], s["std_attack"], s["std_defence"]
        self.standardised_attack, self.standardised_defence = s["standardised_attack"], s["standardised_defence"]
        self.attack_coefficients = s.get("attack_coefficients") if arr.covariates is not None else None
        self.defence_coefficients = s.get("defence_coefficients") if arr.covariates is not None else None
        if self.model == "neutral_wc":
            self.confederation_strength = s["confederation_strength_decentered"]  # LocScaleReparam of N(0,1): identity
            self.conferences, self._conferences_dict = self._meta["conferences"], self._meta["conferences_dict"]
        return self

    def _samples(self):
        d = {"attack": self.attack, "defence": self.defence, "corr_coef": self.corr_coef}
        for nm in self._effects:
            d[nm] = getattr(self, nm)
        return d

    def _fixture_extras(self, n, neutral_venue=0, **kw):
        nv = np.asarray(_str_to_list(neutral_venue)[0], dtype=np.uint8)
        return {"neutral_venue": np.resize(nv, n).astype(np.uint8)}

    def predict_score_proba(self, home_team, away_team, home_goals, away_goals, neutral_venue):
        return super().predict_score_proba(home_team, away_team, home_goals, away_goals, neutral_venue=neutral_venue)

    def predict_score_grid_proba(self, home_team, away_team, neutral_venue, max_goals: int = MAX_GOALS):
        return super().predict_score_grid_proba(home_team, away_team, max_goals=max_goals, neutral_venue=neutral_venue)

    def predict_outcome_proba(self, home_team, away_team, neutral_venue, knockout: bool = False, max_goals: int = MAX_GOALS):
        return super().predict_outcome_proba(home_team, away_team, max_goals=max_goals, knockout=knockout,
                                             neutral_venue=neutral_venue)

    def predict_score_n_proba(self, n, team, opponent, home: bool = True, neutral_venue: int = 0, max_goals: int = MAX_GOALS):
        return self._n_proba(n, team, opponent, home, max_goals, True, neutral_venue=neutral_venue)

    def sample_score(self, home_team, away_team, neutral_venue, num_samples: int = 1, random_state: Optional[int] = None,
                     max_goals: int = MAX_GOALS):
        return self._sample_score(home_team, away_team, num_samples, random_state, max_goals, neutral_venue=neutral_venue)

    def sample_outcome(self, home_team, away_team, neutral_venue, knockout: bool = False, num_samples: int = 1,
                       random_state: Optional[int] = None, max_goals: int = MAX_GOALS):
        return self._sample_outcome(home_team, away_team, num_samples, random_state, max_goals, knockout=knockout,
                                    neutral_venue=neutral_venue)

    def add_new_team(self, team_name: str, team_covariates: Optional[np.ndarray] = None) -> None:
        """``neutral_dixon_coles.py:490-560`` / ``neutral_dixon_coles_WC.py:476-546``: the pair from the correlated prior,
        the four venue effects from their own normal priors."""
        attack, defence = self._new_team_pair(team_name, team_covariates)
        cols = {"attack": attack, "defence": defence}
        for nm in self._effects:
            cols[nm] = np.random.normal(loc=getattr(self, "mean_" + nm), scale=getattr(self, "std_" + nm))
        self._append_team(team_name, cols)

    def predict_concede_n_proba(self, n, team, opponent, home: bool = True, neutral_venue: int = 0,
                                max_goals: int = MAX_GOALS):
        return self._n_proba(n, team, opponent, home, max_goals, False, neutral_venue=neutral_venue)


class NeutralDixonColesMatchPredictorWC(NeutralDixonColesMatchPredictor):
    """``bpl/neutral_dixon_coles_WC.py:31-968``: neutral model + per-confederation strength."""
    model = "neutral_wc"

    def fit(self, training_data, epsilon: float = 0.0, rescale_weights: bool = False, random_state: int = 42,
            num_warmup: int = 500, num_samples: int = 1000, mcmc_kwargs: Optional[Dict[str, Any]] = None,
            run_kwargs: Optional[Dict[str, Any]] = None):
        return super().fit(training_data, epsilon, rescale_weights, random_state, num_warmup, num_samples, mcmc_kwargs,
                           run_kwargs)

    def _samples(self):
        d = super()._samples()
        d["confederation_strength"] = self.confederation_strength
        return d

    def _fixture_extras(self, n, home_conf=None, away_conf=None, neutral_venue=0, **kw):
        out = super()._fixture_extras(n, neutral_venue=neutral_venue)
        for key, val in (("home_conf", home_conf), ("away_conf", away_conf)):
            v = _str_to_list(val)[0]
            if isinstance(v[0], str):
                v = [self._conferences_dict[c] for c in v]
            out[key] = np.resize(np.asarray(v, dtype=np.uint8), n)
        return out

    def predict_score_proba(self, home_team, away_team, home_conf, away_conf, home_goals, away_goals, neutral_venue):
        return _BplxPredictor.predict_score_proba(self, home_team, away_team, home_goals, away_goals, home_conf=home_conf,
                                                  away_conf=away_conf, neutral_venue=neutral_venue)

    def predict_score_grid_proba(self, home_team, away_team, home_conf, away_conf, neutral_venue, max_goals: int = MAX_GOALS):
        return _BplxPredictor.predict_score_grid_proba(self, home_team, away_team, max_goals=max_goals, home_conf=home_conf,
                                                       away_conf=away_conf, neutral_venue=neutral_venue)

    def predict_outcome_proba(self, home_team, away_team, home_conf, away_conf, neutral_venue, knockout: bool = False,
                              max_goals: int = MAX_GOALS):
        return _BplxPredictor.predict_outcome_proba(self, home_team, away_team, max_goals=max_goals, knockout=knockout,
                                                    home_conf=home_conf, away_conf=away_conf, neutral_venue=neutral_venue)

    def sample_score(self, home_team, away_team, home_conf, away_conf, neutral_venue, num_samples: int = 1,
                     random_state: Optional[int] = None, max_goals: int = MAX_GOALS):
        return self._sample_score(home_team, away_team, num_samples, random_state, max_goals, home_conf=home_conf,
                                  away_conf=away_conf, neutral_venue=neutral_venue)

    def sample_outcome(self, home_team, away_team, home_conf, away_conf, neutral_venue, knockout: bool = False,
                       num_samples: int = 1, random_state: Optional[int] = None, max_goals: int = MAX_GOALS):
        return self._sample_outcome(home_team, away_team, num_samples, random_state, max_goals, knockout=knockout,
                                    home_conf=home_conf, away_conf=away_conf, neutral_venue=neutral_venue)

    def _conf_kw(self, team_conf, opponent_conf, home, neutral_venue):
        hc, ac = (team_conf, opponent_conf) if home else (opponent_conf, team_conf)
        return dict(home_conf=hc, away_conf=ac, neutral_venue=neutral_venue)

    def predict_score_n_proba(self, n, team, opponent, team_conf, opponent_conf, home: bool = True, neutral_venue: int = 0,
                              max_goals: int = MAX_GOALS):
        return self._n_proba(n, team, opponent, home, max_goals, True, **self._conf_kw(team_conf, opponent_conf, home, neutral_venue))

    def predict_concede_n_proba(self, n, team, opponent, team_conf, opponent_conf, home: bool = True, neutral_venue: int = 0,
                                max_goals: int = MAX_GOALS):
        return self._n_proba(n, team, opponent, home, max_goals, False, **self._conf_kw(team_conf, opponent_conf, home, neutral_venue))


class DynamicNeutralDixonColesMatchPredictor(_BplxPredictor):
    """``bpl/dynamic_dixon_coles.py:23-334`` -- ``fit`` only.  The reference's predict methods index a Python list with a
    tuple and cannot run (SURVEY.md D3), so they are not mirrored.  ``walk="intended"`` (default) makes attack / defence the
    cumulative random walk the model describes; ``walk="as_written"`` reproduces ``:192-218`` literally (SURVEY D1).
    Gameweeks are 0-based and G = max + 1 (the reference passes ``max``, SURVEY D2)."""
    model = "dynamic"

    def __init__(self, walk: str = "intended"):
        super().__init__()
        if walk not in ("intended", "as_written"):
            raise ValueError(walk)
        self.walk = walk

    def fit(self, training_data, random_state: int = 42, num_warmup: int = 500, num_samples: int = 1000,
            mcmc_kwargs: Optional[Dict[str, Any]] = None, run_kwargs: Optional[Dict[str, Any]] = None):
        kw = dict(mcmc_kwargs or {})
        num_chains = int(kw.pop("num_chains", 1))
        thin = int(kw.pop("thin", kw.pop("thinning", 1)))
        kw.pop("chain_method", None)
        kw.pop("progress_bar", None)
        arr, meta = bdata.prepare("dynamic", training_data)
        arr.as_written = self.walk == "as_written"
        self.teams, self._teams_dict = list(meta["teams"]), meta["teams_dict"]
        self.problem = p = Problem(arr)
        G, T = arr.num_gameweeks, arr.num_teams
        flat_dev, cc = _run_chains(p, num_chains, random_state, num_warmup, num_samples, thin, kw, self)
        flat = flat_dev.cpu().numpy()
        fi = np.finfo(np.float32)
        s = {}
        for name, (off, cnt, tr) in p.layout.items():
            x = flat[:, off:off + cnt]
            if tr == "exp":
                x = np.exp(x)
            elif tr == "sigmoid":
                x = np.clip(1.0 / (1.0 + np.exp(-x)), fi.tiny, 1.0 - fi.eps)
            s[name] = x.astype(np.float32)
        S = flat.shape[0]
        gt = lambda k: s[k].reshape(S, G, T)  # noqa: E731
        self.corr_coef = cc.cpu().numpy()
        self.u, self.rho = gt("u"), 2.0 * gt("u") - 1.0
        self.standardised_attack, self.standardised_defence = gt("standardised_attack"), gt("standardised_defence")
        self.mean_defence = s["mean_defence"][:, 0]
        self.std_attack, self.std_defence = s["std_attack"], s["std_defence"]  # [S, G]
        for nm in ("home_attack", "away_attack", "home_defence", "away_defence"):
            setattr(self, "mean_" + nm, s["mean_" + nm])
            setattr(self, "std_" + nm, s["std_" + nm])
            setattr(self, nm, s["mean_" + nm][:, :, None] + s["std_" + nm][:, :, None] * gt(nm + "_decentered"))
        am, dm = np.zeros((S, 1), np.float32), self.mean_defence[:, None]
        if arr.covariates is not None:
            Xs = arr.covariates.astype(np.float32)
            am, dm = s["attack_coefficients"] @ Xs.T, dm + s["defence_coefficients"] @ Xs.T
            self.attack_coefficients, self.defence_coefficients = s["attack_coefficients"], s["defence_coefficients"]
        else:
            self.attack_coefficients = self.defence_coefficients = None
        step_a = self.standardised_attack * self.std_attack[:, :, None]
        step_d = self.standardised_defence * self.std_defence[:, :, None]
        if self.walk == "intended":
            att, dfn = am[:, None, :] + np.cumsum(step_a, axis=1), dm[:, None, :] + np.cumsum(step_d, axis=1)
        else:  # the recorded deterministics attack_j = 0 + z[j] std[j] for j >= 1 (SURVEY D1)
            att, dfn = step_a.copy(), step_d.copy()
            att[:, 0] += am
            dfn[:, 0] += dm
        self.attack = [att[:, j] for j in range(G)]  # the reference stores lists of [S, T] arrays (:308-309)
        self.defence = [dfn[:, j] for j in range(G)]
        return self

    def simulate_table(self, *args, **kwargs):
        raise NotImplementedError("simulation needs the predictive distribution, and the dynamic model's predict methods "
                                  "cannot run in the reference (SURVEY.md D3)")

    def simulate_tournament(self, *args, **kwargs):
        raise NotImplementedError("simulation needs the predictive distribution, and the dynamic model's predict methods "
                                  "cannot run in the reference (SURVEY.md D3)")

    def posterior_predictive_check(self, *args, **kwargs):
        raise NotImplementedError("posterior predictive checks need the predictive distribution, and the dynamic model's "
                                  "predict methods cannot run in the reference (SURVEY.md D3)")

    def _comparison_inputs(self, data):
        raise NotImplementedError("model comparison needs the predictive distribution, and the dynamic model's predict "
                                  "methods cannot run in the reference (SURVEY.md D3)")
