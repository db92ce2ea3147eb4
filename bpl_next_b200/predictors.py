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
from .problem import Problem, pointwise_loglik, psis_loo, score_grid_host, take_rows
from .problem import simulate_table as _simulate_table
from .problem import simulate_tournament as _simulate_tournament

MAX_GOALS = bdata.MAX_GOALS
# device memory for the [matches, draws] log-likelihood matrix of loo(): larger match sets are processed in ranges
LOO_MATRIX_BYTES = 4 << 30
# device memory for the raw outputs of simulate_table / simulate_tournament(return_simulations=True) (positions, scores,
# knockout entrants, scores and winners): larger runs are processed in ranges of posterior draws
SIM_OUTPUT_BYTES = 1 << 30
# device memory for the [fixtures x markets, draws] matrix of predict_proba_posterior(): larger fixture sets are
# processed in ranges
MARKET_MATRIX_BYTES = 4 << 30
_RATE_ROWS = ("home_rate", "away_rate")


def _half_lines(lines, lo: float, hi: float, what: str) -> list:
    """Validated half-integer lines in [lo, hi] (no pushes), at most ``_abi.MARKET_MAX_LINES``, no repeats."""
    from . import _abi

    out = []
    for x in lines:
        v = float(x) if np.isscalar(x) and not isinstance(x, (bool, np.bool_, str)) else np.nan
        if not np.isfinite(v) or (2.0 * v) % 2.0 != 1.0:
            raise ValueError(f"{what} line {x!r} is not a half-integer (integer and quarter lines are not supported)")
        if not lo <= v <= hi:
            raise ValueError(f"{what} line {v:g} is outside [{lo:g}, {hi:g}] for this max_goals")
        if v in out:
            raise ValueError(f"{what} line {v:g} is given twice")
        out.append(v)
    if len(out) > _abi.MARKET_MAX_LINES:
        raise ValueError(f"at most {_abi.MARKET_MAX_LINES} {what} lines (got {len(out)})")
    return out


def _market_args(total_lines, margin_lines, quantiles, odds, max_goals: int, F: int):
    """Validated lines, levels and odds of ``predict_proba_posterior`` -> (total lines, margin lines, levels, row
    names, odds [F, K] float64 with 0 where a row has none, the names of the rows with odds)."""
    from . import _abi
    from .problem import market_names

    G = int(max_goals)
    if not 1 <= G <= 63:
        raise ValueError(f"max_goals must be in [1, 63] (got {max_goals})")
    tl = _half_lines(total_lines, 0.5, 2 * G - 0.5, "total")
    ml = _half_lines(margin_lines, -G + 0.5, G - 0.5, "margin")
    lv = np.asarray(quantiles, dtype=np.float64).ravel()
    if len(lv) > _abi.QUANTILE_MAX_LEVELS:
        raise ValueError(f"at most {_abi.QUANTILE_MAX_LEVELS} quantile levels (got {len(lv)})")
    if not (np.isfinite(lv) & (lv >= 0.0) & (lv <= 1.0)).all():
        raise ValueError(f"quantile levels must lie in [0, 1] (got {list(lv)})")
    names = market_names(tl, ml)
    om = np.zeros((F, len(names)), np.float64)
    priced = []
    for name, o in (odds or {}).items():
        if name in _RATE_ROWS:
            raise ValueError(f"{name} is an expected number of goals: it takes no odds")
        if name not in names:
            raise ValueError(f"odds for {name!r}, which is not a row of this call (rows: {names})")
        o = np.asarray(o, dtype=np.float64)
        if o.ndim > 1 or (o.ndim == 1 and len(o) != F):
            raise ValueError(f"odds for {name} must be a scalar or one value per fixture ({F})")
        if not (np.isfinite(o) & (o > 1.0)).all():
            raise ValueError(f"odds for {name} must be finite decimal odds > 1")
        om[:, names.index(name)] = o
        priced.append(name)
    return tl, ml, lv, names, om, priced


def _market_result(names, priced, lv, om, S: int, max_goals: int, stats, quant, exceed, draws) -> Dict[str, Any]:
    """The dict ``predict_proba_posterior`` returns, from the per-fixture arrays of ``_market_posterior``."""
    res: Dict[str, Any] = {}
    for k, name in enumerate(names):
        row = {"mean": stats[:, k, 0], "sd": stats[:, k, 1], "quantiles": quant[:, k, :]}
        if name in priced:
            row["edge_proba"] = exceed[:, k] / S
            row["expected_value"] = stats[:, k, 0] * om[:, k] - 1.0
        res[name] = row
    res.update(markets=list(names), quantile_levels=np.asarray(lv, np.float64), num_draws=S, max_goals=int(max_goals))
    if draws is not None:
        res["draws"] = draws
    return res


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

    # ---- forecast uncertainty: the posterior distribution of market probabilities --------------------------------
    @staticmethod
    def _market_posterior(model, samples, fx, max_goals, tl, ml, lv, om, return_draws):
        """Per-draw markets of the fixtures ``fx`` (host index arrays) under the host posterior arrays ``samples``, in
        ranges of fixtures within ``MARKET_MATRIX_BYTES``: (stats [F, K, 2], quantiles [F, K, Q], exceed [F, K] int64,
        draws [F, K, S] or None).  Raises when a draw had a non-finite rate."""
        from .problem import market_draws, row_quantiles

        ds = {k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).cuda() for k, v in samples.items()
              if v is not None}
        dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fx.items()}
        F, K, S, Q = len(fx["home_team"]), om.shape[1], int(ds["attack"].shape[0]), len(lv)
        per = max(1, min(F, MARKET_MATRIX_BYTES // (4 * S * K)))
        buf = torch.empty((per * K, S), dtype=torch.float32, device="cuda")
        dodds = torch.from_numpy(np.ascontiguousarray(om.reshape(-1))).cuda()
        stats, quant = np.empty((F, K, 2)), np.empty((F, K, Q))
        exceed = np.zeros((F, K), np.int64)
        draws = np.empty((F, K, S), np.float32) if return_draws else None
        invalid, ws = 0, None
        for lo in range(0, F, per):
            hi = min(F, lo + per)
            mat, st, inv = market_draws(model, ds, {k: v[lo:hi] for k, v in dfx.items()}, max_goals, tl, ml, draws=buf,
                                        workspace=ws)
            q, e = row_quantiles(mat, lv, dodds[lo * K:hi * K])
            invalid += int(inv.item())
            stats[lo:hi] = st.cpu().numpy().reshape(hi - lo, K, 2)
            quant[lo:hi] = q.cpu().numpy().reshape(hi - lo, K, Q)
            exceed[lo:hi] = e.cpu().numpy().reshape(hi - lo, K)
            if return_draws:
                draws[lo:hi] = mat.cpu().numpy().reshape(hi - lo, K, S)
        if invalid:
            raise ValueError(f"{invalid} of {S * F} (draw, fixture) pairs have a non-finite scoring rate: check the "
                             "posterior draws")
        return stats, quant, exceed, draws

    def _predict_proba_posterior(self, home_team, away_team, total_lines, margin_lines, quantiles, odds, max_goals,
                                 return_draws, **kw):
        fx = self._fixture_arrays(home_team, away_team, kw)
        tl, ml, lv, names, om, priced = _market_args(total_lines, margin_lines, quantiles, odds, max_goals,
                                                     len(fx["home_team"]))
        samples = self._samples()
        stats, quant, exceed, draws = self._market_posterior(self.model, samples, fx, max_goals, tl, ml, lv, om,
                                                             return_draws)
        return _market_result(names, priced, lv, om, int(np.shape(samples["attack"])[0]), max_goals, stats, quant,
                              exceed, draws)

    def predict_proba_posterior(self, home_team, away_team, total_lines=(1.5, 2.5, 3.5), margin_lines=(-1.5, 1.5),
                                quantiles=(0.05, 0.5, 0.95), odds=None, max_goals: int = MAX_GOALS,
                                return_draws: bool = False) -> Dict[str, Any]:
        """Forecast uncertainty: the posterior distribution, over the S draws, of a fixture's market probabilities.

        For draw s the grid is ``P_s(i, j) = tau(i, j) Pois(i; lh_s) Pois(j; la_s)`` for ``0 <= i, j <= max_goals``,
        with the rates of ``predict_*`` (neutral venues and confederations included, no clip), ``c = corr_coef_s`` and
        tau clamped at 0 on the four low cells ((0,0) ``1 - c lh la``, (0,1) ``1 + c lh``, (1,0) ``1 + c la``, (1,1)
        ``1 - c``).  The grid is NOT normalised: these are the cells ``predict_score_grid_proba`` averages, so each
        row's ``mean`` is what the averaged grid gives (``predict_outcome_proba`` for the outcome rows).  Rows per
        fixture, in this order (``markets``): ``home_win``, ``draw``, ``away_win`` (i > j, i = j, i < j);
        ``both_teams_score`` (i >= 1 and j >= 1); ``home_rate``, ``away_rate`` (the rates themselves: expected goals,
        not truncated); per total line L ``total_over_L`` (i + j > L) and ``total_under_L`` (i + j < L); per margin
        line h ``home_margin_over_h`` (i - j > h) and ``home_margin_under_h`` (i - j < h).  Lines are half-integers
        (no pushes): total lines in [0.5, 2 max_goals - 0.5], margin lines in [-max_goals + 0.5, max_goals - 0.5], at
        most 16 of each.  Over and under do not sum to 1 in a draw: the mass beyond ``max_goals`` is dropped, as
        ``predict_score_grid_proba`` drops it.

        Per row: ``mean`` and ``sd`` (divisor S) from float64 sums, ``quantiles [F, Q]`` at ``quantiles`` (numpy's
        ``method="linear"`` on the row's S float32 values, exact order statistics).  ``odds`` maps a row name to
        decimal odds (a scalar or one per fixture; finite, > 1; not the rate rows): the row then also has
        ``edge_proba``, the share of draws with ``p_s * odds > 1`` (in how much of the posterior the bet is worth
        taking), and ``expected_value = mean * odds - 1``.  Also returned: ``markets``, ``quantile_levels``,
        ``num_draws``, ``max_goals``, and with ``return_draws`` the per-draw values ``draws [F, K, S]``.  The fixtures
        run in ranges within ``MARKET_MATRIX_BYTES`` of device memory; the results do not depend on the range size.
        Raises if a draw has a non-finite rate."""
        return self._predict_proba_posterior(home_team, away_team, total_lines, margin_lines, quantiles, odds,
                                             max_goals, return_draws)

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

    def _comparison_inputs(self, data, random_state=None):
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

        seed = int(datetime.now().timestamp() * 100) if random_state is None else int(random_state)
        R, B = int(num_sims_per_draw), int(score_bins)
        if R < 1:
            raise ValueError(f"num_sims_per_draw must be >= 1, got {num_sims_per_draw}")
        ds, do, key = self._comparison_inputs(data, seed)
        S, T, M = int(ds["attack"].shape[-2]), int(ds["attack"].shape[-1]), int(do["home_team"].shape[0])
        step = (2 ** 31 - 1) // R  # replicates per call stay below 2^31
        per_rep = 4 * (B * B + 3 + 3 * T) + 8 * 3 + (2 * M if return_replicates else 0)  # device output bytes
        step = min(step, max(1, SIM_OUTPUT_BYTES // (R * per_rep)))
        parts, scores, invalid = [], [], 0
        for lo in range(0, S, step):
            hi = min(S, lo + step)
            out = self._replicates(ds, do, lo, hi, max_goals, B, points, R, seed, return_replicates)
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

    def _replicates(self, ds, do, lo, hi, max_goals, B, points, R, seed, want_scores):
        """``posterior_predictive`` on draws ``[lo, hi)``."""
        from .problem import posterior_predictive

        return posterior_predictive(self.model, {k: v[lo:hi] for k, v in ds.items()}, do, max_goals, B, points, R, seed,
                                    first_draw=lo, want_scores=want_scores)

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
                       return_simulations: bool = False, tiebreak: str = "goal_difference", key_fixtures=None,
                       events=None) -> Dict[str, Any]:
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
        size.  Raises if any simulation met a non-finite rate.

        Match importance (``key_fixtures`` and ``events``, both or neither): which remaining fixtures decide the title,
        the top four, relegation or who goes through.  ``key_fixtures``: indices into ``fixtures``, in any order and
        any number; ``events``: a mapping label -> ``(team, positions)``, ``positions`` an int or an iterable of 0-based
        positions within the team's group (title: 0; top four: range(4); relegation: (17, 18, 19); through from a
        group: (0, 1)), at most 64 events.  Key fixture j has outcome o in {0 home win, 1 draw, 2 away win} from its
        simulated score; the GPU counts, in the same simulated seasons, how often each outcome occurred and how often
        each event held with it.  Adds ``key_fixtures``, ``events`` (the labels), ``outcome_proba [Kc, 3]``,
        ``event_proba [E]``, ``conditional_proba [Kc, 3, E]`` (P(event | outcome); NaN where the outcome never
        occurred), ``importance [Kc, E]`` (the largest minus the smallest ``conditional_proba`` over the outcomes that
        occurred, 0 if fewer than two did) and the integer ``outcome_counts`` / ``conditional_counts``: a conditional
        probability needs its sample size, and with ``num_sims_per_draw > 1`` the seasons of one draw are correlated,
        so the effective sample size is smaller than the count.  More than 64 key fixtures run in groups of at most 64
        with the same seed, so every group sees the same simulated seasons; each group costs one simulation."""
        if (key_fixtures is None) != (events is None):
            raise ValueError("key_fixtures and events go together: give both or neither")
        home, away = _str_to_list(fixtures["home_team"], fixtures["away_team"])
        tteams = bseason.table_teams(home, away, played, teams)
        table = bseason.build_table(tteams, played, groups, points, tiebreak)
        hs, as_ = bseason.fixture_slots(table, home, away, known_teams=self.teams)
        fx = {**self._fixture_arrays(home, away, fixtures), "home_slot": hs, "away_slot": as_}
        why = "met a non-finite scoring rate or score-grid normaliser: check the posterior draws"
        if key_fixtures is None:
            return self._simulate(table, fx, None, num_sims_per_draw, random_state, max_goals, return_simulations, why)
        cond = bseason.build_conditions(table, len(home), key_fixtures, events)
        if random_state is None:
            random_state = int(datetime.now().timestamp() * 100)  # one seed for every group
        Kc, E = len(cond["key_fixtures"]), len(cond["events"])
        oc, cc = np.zeros((Kc, 3), np.int64), np.zeros((Kc, 3, E), np.int64)
        res = None
        for g in cond["groups"]:
            part = dict(g, event_slot=cond["event_slot"], event_positions=cond["event_positions"])
            out = self._simulate(table, fx, None, num_sims_per_draw, random_state, max_goals,
                                 return_simulations and res is None, why, part)
            oc[g["rows"]], cc[g["rows"]] = out.pop("outcome_counts"), out.pop("conditional_counts")
            res = out if res is None else res
        res.update(bseason.conditional_probabilities(cond, oc, cc, res["num_simulations"]))
        return res

    def _simulate(self, table, fx, bracket, num_sims_per_draw, random_state, max_goals, return_simulations,
                  invalid_reason, conditions=None) -> Dict[str, Any]:
        """``simulate_table`` (``bracket`` None) and ``simulate_tournament`` from the host table, fixture arrays (with
        their slots; ``{}`` for none) and bracket: the draws in ranges, counts summed over the ranges, probabilities.
        With ``conditions`` (one group of ``season.build_conditions``) the result also holds the summed
        ``outcome_counts`` and ``conditional_counts``."""
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
                                      want_positions=return_simulations, want_scores=return_simulations,
                                      conditions=conditions)
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
                                                     cnt["decided_counts"], cnt.get("pairing_counts")))
        res.update({"start_points": table["start_points"].astype(np.int64), "num_simulations": N, "sims_per_draw": R,
                    "seed": seed})
        if conditions is not None:
            res.update(outcome_counts=cnt["outcome_counts"], conditional_counts=cnt["conditional_counts"])
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
                            tiebreak: str = "goal_difference", pairings=None, association=None) -> Dict[str, Any]:
        """A tournament simulated on the GPU: the group stage of ``simulate_table``, then a knockout bracket, with ONE
        posterior draw per simulated tournament, so a team that is stronger in a draw is stronger in every match of its
        path.  (Chaining ``predict_outcome_proba`` calls cannot give this: the opponent of a round depends on earlier
        results, and the same uncertain strengths run through all of a team's matches.)

        ``fixtures``, ``played``, ``teams``, ``groups``, ``points``, ``num_sims_per_draw``, ``random_state``,
        ``max_goals``, ``tiebreak``: as ``simulate_table`` (``"head_to_head"`` ranks each group by the matches among
        its teams level on points, as UEFA's and FIFA's group stages do); ``fixtures`` may be None or empty (a cup: the entrants
        are ``("team", name)``, in fixed ties or in the pools of ``pairings``).  ``bracket``: the ties in play order, ``{"id", "round", "home", "away",
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

        Draws by lot (``pairings``, ``association``; ``season.build_bracket``): domestic cups, the UEFA round of 16,
        open quarter-final draws.  A pairing turns a pool of entrants into pairs when the first tie that takes one of
        its pairs is reached (a tie takes ``"pair": (pairing id, i)`` instead of ``home`` / ``away``), so the opponent
        distribution is part of every simulation.  ``{"id", "pool", "pots": None, ...}`` is an open draw: the pool is
        shuffled and the first team of each pair drawn is at home.  With ``"pots"`` (0 seeded, 1 unseeded, equal in
        size, at most 16 each) it is UEFA's sequential procedure: draw an unseeded team, then one of the seeded teams
        it may meet (``"protect"``: not of the same ``"group"``, not of the same ``"association"``, ``association``
        mapping team -> label) for which the teams left can still be paired; the unseeded team is at home unless
        ``"seeded_home"``.  This is not a uniform choice among the valid pairings, and its pair probabilities differ
        from those.  Adds ``pairing_ids`` and ``pairing_proba [P, T, T]`` (pairing d drew team u at home against team
        v).

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
        named = [e[1] for tie in bracket if "pair" not in tie for e in (tuple(tie["home"]), tuple(tie["away"]))
                 if e[0] == "team"]
        named += [tuple(e)[1] for pg in pairings or () for e in pg["pool"] if tuple(e)[0] == "team"]
        if teams is None:
            tteams = bseason.table_teams(home + named, away, played) if (home or named or played) else []
        else:
            tteams = bseason.table_teams(home, away, played, teams)
        table = bseason.build_table(tteams, played, groups, points, tiebreak)
        br = bseason.build_bracket(table, bracket, best, pairings, association)
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
                              "draws), best-placed qualifiers the bracket does not place, or a pool of a draw "
                              "that could not be paired")

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

    def predict_proba_posterior(self, home_team, away_team, neutral_venue, total_lines=(1.5, 2.5, 3.5),
                                margin_lines=(-1.5, 1.5), quantiles=(0.05, 0.5, 0.95), odds=None,
                                max_goals: int = MAX_GOALS, return_draws: bool = False) -> Dict[str, Any]:
        """The base class's ``predict_proba_posterior`` with ``neutral_venue`` as in ``predict_outcome_proba``."""
        return self._predict_proba_posterior(home_team, away_team, total_lines, margin_lines, quantiles, odds,
                                             max_goals, return_draws, neutral_venue=neutral_venue)

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

    def predict_proba_posterior(self, home_team, away_team, home_conf, away_conf, neutral_venue,
                                total_lines=(1.5, 2.5, 3.5), margin_lines=(-1.5, 1.5), quantiles=(0.05, 0.5, 0.95),
                                odds=None, max_goals: int = MAX_GOALS, return_draws: bool = False) -> Dict[str, Any]:
        """The base class's ``predict_proba_posterior`` with the fixture arguments of ``predict_outcome_proba``."""
        return self._predict_proba_posterior(home_team, away_team, total_lines, margin_lines, quantiles, odds,
                                             max_goals, return_draws, home_conf=home_conf, away_conf=away_conf,
                                             neutral_venue=neutral_venue)

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
    """``bpl/dynamic_dixon_coles.py:23-334``.  ``walk="intended"`` (default) makes attack / defence the cumulative random
    walk the model describes; ``walk="as_written"`` reproduces ``:192-218`` literally (SURVEY D1).  Gameweeks are 0-based
    and G = max + 1 (the reference passes ``max``, SURVEY D2).

    Predictive distribution.  The reference's predict methods index a Python list with a tuple and cannot run (SURVEY
    D3), and their venue signs disagree with ``_model``; they are not mirrored.  Instead, at a fixed gameweek the model's
    rates are exactly the NEUTRAL model's rates, so every predictive method works on one gameweek of the posterior at a
    time (``at_gameweek``), with the rates of ``_model``:

    * Scope: only a fit with ``walk="intended"`` has a predictive distribution (an ``as_written`` fit's likelihood never
      reaches the walk); otherwise every predictive method raises ``NotImplementedError``.
    * Fitted gameweek (g < G): per draw, ``attack[g]``, ``defence[g]``, the four venue effects ``[:, g]`` and
      ``corr_coef``, as ``fit`` records them.
    * Forecast gameweek (g >= G): the model's own generative process continued from the last fitted state.  For each
      draw and each gameweek j = G .. g in order, fresh sites from their priors (means N(+-0.1, 0.2), the six spreads
      HalfNormal(1), per team u ~ Beta(2, 4), rho = 2u - 1, za ~ N(0, 1), zd = rho za + sqrt(1 - rho^2) eps, the four
      decentred effects N(0, 1)); ``attack[j] = attack[j - 1] + za std_attack[j]`` (defence likewise with zd), venue
      effects ``mean[j] + std[j] decentered[j]`` (not cumulative).  With HalfNormal(1) venue spreads this forecast is
      WIDE: it is what the model says about gameweeks it has not seen, nothing more.  Its random numbers are Philox words
      under ``random_state`` (include/bplx.h gives the word map), the same for any cut of the draws.
    * ``gameweek`` defaults to G - 1, the latest fitted state (not a forecast).
    """
    model = "dynamic"
    _effects = NeutralDixonColesMatchPredictor._effects
    _fixture_extras = NeutralDixonColesMatchPredictor._fixture_extras

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
        self._train_arrays = arr  # the matches log_likelihood() / waic() / loo() evaluate by default
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

    # ---- the predictive distribution: one gameweek of the posterior is a NEUTRAL sample set ----------------------
    def _require_predictive(self):
        if getattr(self, "attack", None) is None or self.walk != "intended":
            raise NotImplementedError(
                "the dynamic model's predictive distribution needs a fit of a predictor built with walk=\"intended\" "
                "(the constructor argument): an as_written fit's likelihood never reaches the walk (SURVEY D1)")

    @staticmethod
    def _seed(random_state) -> int:
        return int(datetime.now().timestamp() * 100) if random_state is None else int(random_state)

    def _fixture_gameweeks(self, gameweek, n: int) -> np.ndarray:
        """``[n]`` gameweeks of the fixtures: None -> G - 1, a scalar for all, or one per fixture."""
        if gameweek is None:
            return np.full(n, len(self.attack) - 1, np.int64)
        g = np.asarray(gameweek)
        if g.dtype.kind not in "iu" or (g.ndim == 1 and len(g) not in (1, n)) or g.ndim > 1:
            raise ValueError(f"gameweek must be an integer or one integer per fixture (got {gameweek!r})")
        if (g < 0).any():
            raise ValueError(f"gameweek must be >= 0 (got {gameweek!r})")
        return np.resize(g.astype(np.int64), n)

    def _one_gameweek(self, gameweek) -> int:
        if np.ndim(gameweek) > 0:
            if len(np.unique(np.asarray(gameweek))) != 1:
                raise ValueError("every fixture of this call is played at one gameweek: pass a single gameweek")
            gameweek = np.asarray(gameweek)[0]
        return int(self._fixture_gameweeks(gameweek, 1)[0])

    def _slabs(self, gameweeks, seed: int) -> Dict[int, Dict[str, np.ndarray]]:
        """NEUTRAL sample sets ``{g: {attack, defence, four venue effects [S, T], corr_coef [S]}}`` of the gameweeks, the
        forecast ones drawn in one call under ``seed``."""
        from .problem import dynamic_forecast

        G = len(self.attack)
        gws = sorted({int(g) for g in gameweeks})
        fc = None
        if gws and gws[-1] >= G:
            dev = lambda x: torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()  # noqa: E731
            out = dynamic_forecast(dev(self.attack[G - 1]), dev(self.defence[G - 1]), gws[-1] - G + 1, seed)
            fc = {k: v.cpu().numpy() for k, v in out.items()}
        slabs = {}
        for g in gws:
            if g < G:
                d = {"attack": self.attack[g], "defence": self.defence[g],
                     **{nm: getattr(self, nm)[:, g] for nm in self._effects}}
            else:
                d = {k: fc[k][g - G] for k in fc}
            d = {k: np.ascontiguousarray(v, np.float32) for k, v in d.items()}
            d["corr_coef"] = np.ascontiguousarray(self.corr_coef, np.float32)
            slabs[g] = d
        return slabs

    def at_gameweek(self, gameweek: int, random_state: int = 0) -> "NeutralDixonColesMatchPredictor":
        """A ``NeutralDixonColesMatchPredictor`` with the same teams and this gameweek's draws (fitted for g < G, else
        the forecast under ``random_state``): every single-gameweek question goes through the NEUTRAL class."""
        self._require_predictive()
        g = self._one_gameweek(gameweek)
        p = NeutralDixonColesMatchPredictor()
        p.teams, p._teams_dict = list(self.teams), dict(self._teams_dict)
        for k, v in self._slabs([g], self._seed(random_state))[g].items():
            setattr(p, k, v)
        return p

    def _grid(self, home_team, away_team, max_goals, gameweek=None, forecast_seed=0, **kw):
        """The base class's grid, per fixture at its gameweek: the fixtures are grouped by gameweek, each group through
        the NEUTRAL grid of that gameweek's draws."""
        h, a = self._parse_fixture_args(home_team, away_team)
        fx = {"home_team": h, "away_team": a, **self._fixture_extras(len(h), **kw)}
        gw = self._fixture_gameweeks(gameweek, len(h))
        g = max_goals + 1
        grid, outcome = np.empty((len(h), g, g), np.float32), np.empty((len(h), 3), np.float32)
        for gv, smp in self._slabs(np.unique(gw), int(forecast_seed)).items():
            idx = np.flatnonzero(gw == gv)
            grid[idx], outcome[idx] = score_grid_host("neutral", smp, {k: v[idx] for k, v in fx.items()}, max_goals)
        return grid, outcome

    def predict_score_grid_proba(self, home_team, away_team, neutral_venue, max_goals: int = MAX_GOALS, gameweek=None,
                                 random_state: int = 0):
        """NEUTRAL's ``predict_score_grid_proba`` at ``gameweek`` (scalar or per fixture; default G - 1); forecast
        gameweeks under ``random_state``."""
        self._require_predictive()
        return _BplxPredictor.predict_score_grid_proba(self, home_team, away_team, max_goals=max_goals,
                                                       neutral_venue=neutral_venue, gameweek=gameweek,
                                                       forecast_seed=random_state)

    def predict_outcome_proba(self, home_team, away_team, neutral_venue, knockout: bool = False,
                              max_goals: int = MAX_GOALS, gameweek=None, random_state: int = 0):
        """NEUTRAL's ``predict_outcome_proba`` at ``gameweek`` (see ``predict_score_grid_proba``)."""
        self._require_predictive()
        return _BplxPredictor.predict_outcome_proba(self, home_team, away_team, max_goals=max_goals, knockout=knockout,
                                                    neutral_venue=neutral_venue, gameweek=gameweek,
                                                    forecast_seed=random_state)

    def predict_score_proba(self, home_team, away_team, home_goals, away_goals, neutral_venue, gameweek=None,
                            random_state: int = 0):
        """NEUTRAL's ``predict_score_proba`` at ``gameweek`` (see ``predict_score_grid_proba``)."""
        self._require_predictive()
        return _BplxPredictor.predict_score_proba(self, home_team, away_team, home_goals, away_goals,
                                                  neutral_venue=neutral_venue, gameweek=gameweek,
                                                  forecast_seed=random_state)

    def predict_proba_posterior(self, home_team, away_team, neutral_venue, total_lines=(1.5, 2.5, 3.5),
                                margin_lines=(-1.5, 1.5), quantiles=(0.05, 0.5, 0.95), odds=None,
                                max_goals: int = MAX_GOALS, return_draws: bool = False, gameweek=None,
                                random_state: int = 0) -> Dict[str, Any]:
        """NEUTRAL's ``predict_proba_posterior`` at ``gameweek`` (scalar or per fixture; default G - 1), forecast
        gameweeks under ``random_state``: the fixtures are grouped by gameweek, each group on that gameweek's draws, so
        every fixture's result is the bits of ``at_gameweek(g, random_state).predict_proba_posterior(...)``."""
        self._require_predictive()
        fx = self._fixture_arrays(home_team, away_team, {"neutral_venue": neutral_venue})
        F = len(fx["home_team"])
        gw = self._fixture_gameweeks(gameweek, F)
        tl, ml, lv, names, om, priced = _market_args(total_lines, margin_lines, quantiles, odds, max_goals, F)
        S, K = len(self.corr_coef), len(names)
        stats, quant, exceed = np.empty((F, K, 2)), np.empty((F, K, len(lv))), np.zeros((F, K), np.int64)
        draws = np.empty((F, K, S), np.float32) if return_draws else None
        for gv, smp in self._slabs(np.unique(gw), int(random_state)).items():
            idx = np.flatnonzero(gw == gv)
            part = self._market_posterior("neutral", smp, {k: v[idx] for k, v in fx.items()}, max_goals, tl, ml, lv,
                                          om[idx], return_draws)
            stats[idx], quant[idx], exceed[idx] = part[:3]
            if return_draws:
                draws[idx] = part[3]
        return _market_result(names, priced, lv, om, S, max_goals, stats, quant, exceed, draws)

    def predict_score_n_proba(self, n, team, opponent, home: bool = True, neutral_venue: int = 0,
                              max_goals: int = MAX_GOALS, gameweek=None, random_state: int = 0):
        self._require_predictive()
        return self._n_proba(n, team, opponent, home, max_goals, True, neutral_venue=neutral_venue,
                             gameweek=self._one_gameweek(gameweek), forecast_seed=random_state)

    def predict_concede_n_proba(self, n, team, opponent, home: bool = True, neutral_venue: int = 0,
                                max_goals: int = MAX_GOALS, gameweek=None, random_state: int = 0):
        self._require_predictive()
        return self._n_proba(n, team, opponent, home, max_goals, False, neutral_venue=neutral_venue,
                             gameweek=self._one_gameweek(gameweek), forecast_seed=random_state)

    def sample_score(self, home_team, away_team, neutral_venue, num_samples: int = 1, random_state: Optional[int] = None,
                     max_goals: int = MAX_GOALS, gameweek=None):
        """NEUTRAL's ``sample_score`` at ``gameweek``; ``random_state`` seeds both the forecast and the sampling."""
        self._require_predictive()
        seed = self._seed(random_state)
        return self._sample_score(home_team, away_team, num_samples, seed, max_goals, neutral_venue=neutral_venue,
                                  gameweek=gameweek, forecast_seed=seed)

    def sample_outcome(self, home_team, away_team, neutral_venue, knockout: bool = False, num_samples: int = 1,
                       random_state: Optional[int] = None, max_goals: int = MAX_GOALS, gameweek=None):
        """NEUTRAL's ``sample_outcome`` at ``gameweek``; ``random_state`` seeds both the forecast and the sampling."""
        self._require_predictive()
        seed = self._seed(random_state)
        return self._sample_outcome(home_team, away_team, num_samples, seed, max_goals, knockout=knockout,
                                    neutral_venue=neutral_venue, gameweek=gameweek, forecast_seed=seed)

    def simulate_table(self, fixtures, played=None, teams=None, groups=None, num_sims_per_draw: int = 1,
                       random_state: Optional[int] = None, max_goals: int = MAX_GOALS, points=(3, 1),
                       return_simulations: bool = False, tiebreak: str = "goal_difference", gameweek=None,
                       key_fixtures=None, events=None):
        """NEUTRAL's ``simulate_table`` with every fixture played at one ``gameweek`` (default G - 1; "the next season"
        is ``gameweek=G`` when the gameweeks are seasons).  ``random_state`` seeds the forecast and the simulation;
        ``key_fixtures`` / ``events`` give match importance as there."""
        self._require_predictive()
        seed = self._seed(random_state)
        return self.at_gameweek(self._one_gameweek(gameweek), seed).simulate_table(
            fixtures, played, teams, groups, num_sims_per_draw, seed, max_goals, points, return_simulations, tiebreak,
            key_fixtures, events)

    def simulate_tournament(self, fixtures, bracket, played=None, teams=None, groups=None, best=None, team_conf=None,
                            num_sims_per_draw: int = 1, random_state: Optional[int] = None, max_goals: int = MAX_GOALS,
                            points=(3, 1), return_simulations: bool = False, tiebreak: str = "goal_difference",
                            pairings=None, association=None, gameweek=None):
        """NEUTRAL's ``simulate_tournament`` with every match played at one ``gameweek`` (see ``simulate_table``)."""
        self._require_predictive()
        seed = self._seed(random_state)
        return self.at_gameweek(self._one_gameweek(gameweek), seed).simulate_tournament(
            fixtures, bracket, played, teams, groups, best, team_conf, num_sims_per_draw, seed, max_goals, points,
            return_simulations, tiebreak, pairings, association)

    # ---- model comparison and predictive checks over the gameweeks of the data --------------------------------------
    def _comparison_inputs(self, data, random_state=0):
        """Device samples ``[G', S, T]`` of the gameweeks the matches of ``data`` (default: the training data) use, the
        device observations with ``gameweek`` (host, each match's index into the G' gameweeks) and the match key."""
        self._require_predictive()
        obs, key = self._observations(data)
        if data is None:
            gw = np.asarray(self._train_arrays.gameweek, np.int64)
            obs.setdefault("neutral_venue", np.zeros(len(gw), np.uint8))
        else:
            if "gameweek" not in data:
                raise ValueError("the dynamic model scores each match at its gameweek: data needs the key 'gameweek'")
            gw = self._fixture_gameweeks(np.asarray(data["gameweek"]), len(obs["home_team"]))
        used, index = np.unique(gw, return_inverse=True)
        slabs = self._slabs(used, self._seed(random_state))
        ds = {k: torch.from_numpy(np.stack([slabs[g][k] for g in used])).cuda() for k in slabs[int(used[0])]}
        do = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in obs.items()}
        do["gameweek"] = index.astype(np.int32)
        return ds, do, key

    def _pointwise(self, ds, do, **kw):
        from .problem import pointwise_loglik_gameweeks

        dev = {k: v for k, v in do.items() if k != "gameweek"}
        return pointwise_loglik_gameweeks("neutral", ds, dev, do["gameweek"], **kw)

    def log_likelihood(self, data=None, random_state: int = 0) -> np.ndarray:
        """The base class's ``log_likelihood`` with each match scored at its gameweek (``data["gameweek"]``; held-out
        gameweeks >= G on the forecast under ``random_state``), in one launch over all gameweeks."""
        ds, do, _ = self._comparison_inputs(data, random_state)
        ll, _ = self._pointwise(ds, do)
        return np.ascontiguousarray(ll.cpu().numpy().T)

    def waic(self, data=None, random_state: int = 0) -> Dict[str, Any]:
        """The base class's ``waic`` with each match scored at its gameweek (see ``log_likelihood``)."""
        ds, do, key = self._comparison_inputs(data, random_state)
        _, st = self._pointwise(ds, do, want_matrix=False)
        return bcompare.waic_from_stats(st.cpu().numpy(), int(ds["attack"].shape[1]), key)

    def log_score(self, data, random_state: int = 0) -> Dict[str, Any]:
        """The base class's ``log_score`` with each match scored at its gameweek: later gameweeks (>= G) on the forecast
        under ``random_state``, so "does the walk forecast the next season better than a static fit?" is one comparison
        of the two log scores."""
        ds, do, _ = self._comparison_inputs(data, random_state)
        _, st = self._pointwise(ds, do, want_matrix=False)
        lppd = bcompare.lppd_from_stats(st.cpu().numpy(), int(ds["attack"].shape[1]))
        return {"log_score": float(lppd.sum()), "pointwise": lppd, "num_matches": len(lppd)}

    def loo(self, r_eff: float = 1.0) -> Dict[str, Any]:
        """The base class's ``loo`` on the training data, each match scored at its (fitted) gameweek: the matrix of the
        matches grouped by gameweek comes from one launch per range of ``LOO_MATRIX_BYTES``; results in match order."""
        ds, do, key = self._comparison_inputs(None)
        S, M = int(ds["attack"].shape[1]), int(do["home_team"].shape[0])
        order = np.argsort(do["gameweek"], kind="stable")
        idx = torch.from_numpy(order).cuda()
        srt = {k: (v[order] if k == "gameweek" else take_rows(v, idx)) for k, v in do.items()}
        rows = max(1, min(M, LOO_MATRIX_BYTES // (4 * S)))
        buf = torch.empty((rows, S), dtype=torch.float32, device="cuda")
        elpd, khat, lppd = [], [], []
        for lo in range(0, M, rows):
            hi = min(M, lo + rows)
            ll, st = self._pointwise(ds, {k: v[lo:hi] for k, v in srt.items()}, loglik=buf)
            e, k = psis_loo(ll, r_eff)
            elpd.append(e.cpu().numpy())
            khat.append(k.cpu().numpy())
            lppd.append(bcompare.lppd_from_stats(st.cpu().numpy(), S))
        inv = np.argsort(order, kind="stable")
        return bcompare.loo_from_pointwise(np.concatenate(elpd)[inv], np.concatenate(khat)[inv],
                                           np.concatenate(lppd)[inv], S, r_eff, key)

    def posterior_predictive_check(self, data=None, num_sims_per_draw: int = 1, random_state: Optional[int] = None,
                                   max_goals: int = MAX_GOALS, score_bins: int = 6, points=(3, 1),
                                   return_replicates: bool = False) -> Dict[str, Any]:
        """The base class's ``posterior_predictive_check`` with each match replicated at its gameweek
        (``data["gameweek"]``, default the training data; ``random_state`` also seeds forecast gameweeks): the same
        replicate index, words and statistics, one launch per range of draws."""
        self._require_predictive()
        return super().posterior_predictive_check(data, num_sims_per_draw, random_state, max_goals, score_bins, points,
                                                  return_replicates)

    def _replicates(self, ds, do, lo, hi, max_goals, B, points, R, seed, want_scores):
        from .problem import posterior_predictive_gameweeks

        dev = {k: v for k, v in do.items() if k != "gameweek"}
        return posterior_predictive_gameweeks("neutral", {k: v[:, lo:hi].contiguous() for k, v in ds.items()}, dev,
                                              do["gameweek"], max_goals, B, points, R, seed, first_draw=lo,
                                              want_scores=want_scores)
