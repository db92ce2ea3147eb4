"""Python handles over the C ABI: ``Problem`` (log-density + gradient), ``score_grid``, ``pointwise_loglik``,
``psis_loo``, ``simulate_table``, ``simulate_tournament``, ``posterior_predictive``, ``market_draws`` and
``row_quantiles``; for the dynamic model's gameweeks ``dynamic_forecast``, ``pointwise_loglik_gameweeks`` and
``posterior_predictive_gameweeks``.

torch is used only for device memory and streams; every number comes from ``libbplx.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _abi
from .data import MatchArrays
from .season import TIEBREAKS

_STAT_NAMES = ("matches", "entries1", "entries1_padded", "entries2", "entries2_padded", "smem_bytes", "warps", "vteams")


def _stream_ptr(stream=None) -> int:
    s = stream if stream is not None else torch.cuda.current_stream()
    return int(s.cuda_stream)


def _dptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else int(t.data_ptr())


class Problem:
    """Static match data bound to the current CUDA device (``bplx_problem``)."""

    def __init__(self, arrays: MatchArrays):
        if not torch.cuda.is_available():
            raise RuntimeError("bpl_next_b200 needs a CUDA device: there is no CPU fallback")
        self._lib = _abi.lib()
        self.arrays = arrays
        self._h = C.c_void_p()
        desc = arrays.desc()
        torch.cuda.current_device()  # make sure the primary context exists
        _abi.check(self._lib.bplx_problem_create(C.byref(desc), C.byref(self._h)))
        self.D = int(self._lib.bplx_num_params(self._h))
        self.layout = self._parse_layout(self._lib.bplx_problem_layout(self._h).decode())
        self._ws: Optional[torch.Tensor] = None

    @staticmethod
    def _parse_layout(s: str) -> Dict[str, Tuple[int, int, str]]:
        out = {}
        for rec in filter(None, s.split(";")):
            name, off, cnt, tr = rec.split(":")
            out[name] = (int(off), int(cnt), tr)
        return out

    def stats(self) -> Dict[str, int]:
        buf = (C.c_longlong * 8)()
        self._lib.bplx_problem_stats(self._h, buf, 8)
        return dict(zip(_STAT_NAMES, [int(x) for x in buf]))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.bplx_problem_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- device path -------------------------------------------------------------------------
    def workspace(self, num_chains: int) -> Optional[torch.Tensor]:
        need = int(self._lib.bplx_logdensity_workspace_bytes(self._h, num_chains))
        if need == 0:
            return None
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        return self._ws

    def logdensity(self, theta: torch.Tensor, chain_minor: bool = False, lp=None, grad=None, corr_coef=None,
                   stream=None):
        """Enqueue log-density + gradient.  ``theta`` is ``[C, D]`` (chain-major) or ``[D, C]``
        (``chain_minor=True``), float32, on the GPU; rows may be padded (a view with unit inner stride: the row pitch is
        passed as the leading dimension, and ``grad`` must have the same pitch).  Returns ``(lp, grad, corr_coef)``."""
        assert theta.is_cuda and theta.dtype == torch.float32 and theta.dim() == 2
        assert theta.stride(1) == 1 or theta.shape[1] == 1  # (the stride of a one-element dimension means nothing)
        if chain_minor:
            D, Cn = theta.shape
        else:
            Cn, D = theta.shape
        if D != self.D:
            raise ValueError(f"theta has {D} parameters, the model has {self.D}")
        lp = torch.empty(Cn, dtype=torch.float32, device=theta.device) if lp is None else lp
        grad = torch.empty_strided(theta.shape, theta.stride(), dtype=torch.float32, device=theta.device) if grad is None else grad
        assert grad.shape == theta.shape and grad.stride() == theta.stride()
        corr_coef = torch.empty(Cn, dtype=torch.float32, device=theta.device) if corr_coef is None else corr_coef
        ws = self.workspace(Cn)
        ld = int(theta.stride(0)) if theta.shape[0] > 1 else 0
        _abi.check(self._lib.bplx_logdensity_fwdbwd(
            self._h, Cn, _abi.CHAIN_MINOR if chain_minor else _abi.CHAIN_MAJOR, ld,
            _dptr(theta), _dptr(lp), _dptr(grad), _dptr(corr_coef),
            _dptr(ws), 0 if ws is None else ws.numel(), _stream_ptr(stream)))
        return lp, grad, corr_coef

    # ---- likelihood-only entry (what a numpyro model that keeps its prior sites hands to numpyro.factor) -------
    @property
    def loglik_layout(self) -> Dict[str, Tuple[int, int, str]]:
        return self._parse_layout(self._lib.bplx_loglik_layout(self._h).decode())

    def loglik(self, tables: torch.Tensor, chain_minor: bool = False, stream=None):
        """``tables``: the constrained per-team tables packed per ``loglik_layout`` (``[C, Dl]`` or ``[Dl, C]``).
        Returns ``(loglik [C], grad (like tables), corr_coef [C])``: Poisson + tau terms only, no priors."""
        assert tables.is_cuda and tables.dtype == torch.float32 and tables.is_contiguous()
        Dl = int(self._lib.bplx_loglik_num_inputs(self._h))
        if Dl < 0:
            _abi.check(Dl)
        Cn = tables.shape[1] if chain_minor else tables.shape[0]
        if (tables.shape[0] if chain_minor else tables.shape[1]) != Dl:
            raise ValueError(f"tables have {tables.shape} entries, the likelihood takes {Dl} per chain")
        ll = torch.empty(Cn, dtype=torch.float32, device=tables.device)
        grad = torch.empty_like(tables)
        cc = torch.empty(Cn, dtype=torch.float32, device=tables.device)
        ws = self.workspace(Cn)
        _abi.check(self._lib.bplx_loglik_fwdbwd(
            self._h, Cn, _abi.CHAIN_MINOR if chain_minor else _abi.CHAIN_MAJOR, 0, _dptr(tables), _dptr(ll),
            _dptr(grad), _dptr(cc), _dptr(ws), 0 if ws is None else ws.numel(), _stream_ptr(stream)))
        return ll, grad, cc

    # ---- host path (the reference-facing call: numpy in, numpy out) --------------------------------
    def logdensity_host(self, theta: np.ndarray, lp=None, grad=None, corr_coef=None):
        theta = np.ascontiguousarray(theta, dtype=np.float32)
        Cn, D = theta.shape
        if D != self.D:
            raise ValueError(f"theta has {D} parameters, the model has {self.D}")
        lp = np.empty(Cn, dtype=np.float32) if lp is None else lp
        grad = np.empty((Cn, D), dtype=np.float32) if grad is None else grad
        corr_coef = np.empty(Cn, dtype=np.float32) if corr_coef is None else corr_coef
        _abi.check(self._lib.bplx_logdensity_fwdbwd_host(self._h, Cn, theta.ctypes.data, lp.ctypes.data,
                                                         grad.ctypes.data, corr_coef.ctypes.data))
        return lp, grad, corr_coef


# ------------------------------------------------------------------------------------------------------
_SAMPLE_KEYS = ("attack", "defence", "home_attack", "away_attack", "home_defence", "away_defence",
                "confederation_strength", "corr_coef")
_FIXTURE_KEYS = (("home_team", np.uint16), ("away_team", np.uint16), ("home_conf", np.uint8),
                 ("away_conf", np.uint8), ("neutral_venue", np.uint8))


def _samples_struct(model: str, samples: dict, ptr):
    s = _abi.Samples()
    s.model = _abi.MODEL_IDS[model]
    att = samples["attack"]
    s.num_samples, s.num_teams = int(att.shape[0]), int(att.shape[1])
    cs = samples.get("confederation_strength")
    s.num_conferences = 0 if cs is None else int(cs.shape[1])
    src = dict(samples)
    if model in ("dixon_coles", "extended"):
        src["home_attack"] = samples["home_advantage"]  # include/bplx.h: home advantage travels here
    for k in _SAMPLE_KEYS:
        v = src.get(k)
        setattr(s, k, None if v is None else ptr(v))
    return s


def _fixtures_struct(fixtures: dict, ptr):
    f = _abi.Fixtures()
    f.num_fixtures = int(len(fixtures["home_team"]))
    for k, _ in _FIXTURE_KEYS:
        v = fixtures.get(k)
        setattr(f, k, None if v is None else ptr(v))
    return f


def _device_ptr_fn(keep):
    def ptr(t):
        assert t.is_cuda and t.is_contiguous()
        keep.append(t)
        return int(t.data_ptr())
    return ptr


def _check_inputs(samples: dict, fixtures: dict, uint8_keys=()):
    """dtypes of device inputs: float32 samples, uint16 / uint8 fixture indices, and ``fixtures[k]`` uint8 for every k
    of ``uint8_keys``."""
    for k in _SAMPLE_KEYS + ("home_advantage",):
        if samples.get(k) is not None:
            assert samples[k].dtype == torch.float32
    for k, dt in _FIXTURE_KEYS:
        if fixtures.get(k) is not None:
            assert fixtures[k].dtype == (torch.uint16 if dt == np.uint16 else torch.uint8), k
    for k in uint8_keys:
        assert fixtures[k].dtype == torch.uint8, k


def _workspace(workspace, need: int, device):
    """``workspace`` when it holds ``need`` bytes, else a new device buffer."""
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(max(need, 1), dtype=torch.uint8, device=device)
    return workspace


def _observations_struct(observations: dict, ptr):
    o = _abi.Observations()
    o.fixtures = _fixtures_struct(observations, ptr)
    o.home_goals, o.away_goals = ptr(observations["home_goals"]), ptr(observations["away_goals"])
    return o


def _output_matrix(buf: Optional[torch.Tensor], rows: int, S: int, device, want: bool):
    """``(matrix, ld)``: the ``[rows, ld]`` float32 output (``buf``, else a new ``[rows, S]`` one) or ``(None, 0)``."""
    if not want:
        return None, 0
    if buf is None:
        buf = torch.empty((rows, S), dtype=torch.float32, device=device)
    assert buf.dtype == torch.float32 and buf.shape[0] >= rows and buf.stride(1) == 1
    return buf, int(buf.stride(0)) if rows > 1 else max(S, int(buf.shape[1]))


def _ppc_outputs(N: int, M: int, T: int, B: int, device, want_scores: bool):
    """Outputs of a predictive check (N replicates, M matches, T teams, B score bins) and their ``_abi.PpcOutput``."""
    i32, i64 = dict(dtype=torch.int32, device=device), dict(dtype=torch.int64, device=device)
    shapes = {"score_counts": ((N, B, B), i32), "outcome_counts": ((N, 3), i32), "goals": ((N, 2), i64),
              "total_goals_sq": ((N,), i64), "team_points": ((N, T), i32), "team_goals_for": ((N, T), i32),
              "team_goals_against": ((N, T), i32)}
    res = {k: torch.empty(shp, **kw) for k, (shp, kw) in shapes.items()}
    res["invalid"] = torch.empty(1, **i64)
    res["scores"] = torch.empty((N, M, 2), dtype=torch.uint8, device=device) if want_scores else None
    return res, _abi.PpcOutput(**{k: _dptr(v) for k, v in res.items()})


def _seed(seed: int) -> int:
    """The 64-bit seed the C ABI takes (``unsigned long long``) of a Python int."""
    return int(seed) & 0xFFFFFFFFFFFFFFFF


def score_grid_workspace_bytes(model: str, samples: Dict[str, torch.Tensor], fixtures: Dict[str, torch.Tensor],
                               max_goals: int) -> int:
    """Bytes of device workspace ``score_grid`` needs for these shapes (``bplx_score_grid_workspace_bytes``)."""
    lib = _abi.lib()
    s = _samples_struct(model, samples, lambda t: int(t.data_ptr()))
    f = _fixtures_struct(fixtures, lambda t: int(t.data_ptr()))
    return int(lib.bplx_score_grid_workspace_bytes(C.byref(s), C.byref(f), max_goals))


def score_grid(model: str, samples: Dict[str, torch.Tensor], fixtures: Dict[str, torch.Tensor], max_goals: int,
               scale: Optional[float] = None, want_outcome: bool = True, workspace=None, grid=None, outcome=None,
               stream=None, reuse_tables: bool = False):
    """Device path: posterior arrays ``[S, T]`` float32 and fixture index tensors on the GPU.
    Returns ``(grid [F, g, g], outcome [F, 3] or None)``; ``scale`` defaults to ``1/S``.  ``reuse_tables``: the
    ``workspace`` passed in still holds the exponential tables a previous call built from these very samples."""
    lib = _abi.lib()
    keep = []
    ptr = _device_ptr_fn(keep)
    _check_inputs(samples, fixtures)
    s = _samples_struct(model, samples, ptr)
    f = _fixtures_struct(fixtures, ptr)
    g = max_goals + 1
    dev = samples["attack"].device
    workspace = _workspace(workspace, int(lib.bplx_score_grid_workspace_bytes(C.byref(s), C.byref(f), max_goals)), dev)
    grid = torch.empty((f.num_fixtures, g, g), dtype=torch.float32, device=dev) if grid is None else grid
    if want_outcome and outcome is None:
        outcome = torch.empty((f.num_fixtures, 3), dtype=torch.float32, device=dev)
    scale = 1.0 / s.num_samples if scale is None else scale
    _abi.check(lib.bplx_score_grid_ex(C.byref(s), C.byref(f), max_goals, C.c_float(scale), _dptr(grid),
                                      _dptr(outcome) if want_outcome else None, _dptr(workspace), workspace.numel(),
                                      _stream_ptr(stream), 1 if reuse_tables else 0))
    return grid, (outcome if want_outcome else None)


def score_grid_host(model: str, samples: Dict[str, np.ndarray], fixtures: Dict[str, np.ndarray], max_goals: int,
                    scale: Optional[float] = None, want_outcome: bool = True):
    """Host path: numpy in, numpy out (copies inside the call)."""
    lib = _abi.lib()
    keep = []

    def ptr(a):
        keep.append(a)
        return a.ctypes.data

    smp = {k: (None if v is None else np.ascontiguousarray(v, dtype=np.float32)) for k, v in samples.items()}
    fx = {k: (None if fixtures.get(k) is None else np.ascontiguousarray(fixtures[k], dtype=dt)) for k, dt in _FIXTURE_KEYS}
    s = _samples_struct(model, smp, ptr)
    f = _fixtures_struct(fx, ptr)
    g = max_goals + 1
    grid = np.empty((f.num_fixtures, g, g), dtype=np.float32)
    outcome = np.empty((f.num_fixtures, 3), dtype=np.float32) if want_outcome else None
    scale = 1.0 / s.num_samples if scale is None else scale
    _abi.check(lib.bplx_score_grid_host(C.byref(s), C.byref(f), max_goals, C.c_float(scale), grid.ctypes.data,
                                        None if outcome is None else outcome.ctypes.data))
    return grid, outcome


def pointwise_loglik(model: str, samples: Dict[str, torch.Tensor], observations: Dict[str, torch.Tensor],
                     want_matrix: bool = True, loglik: Optional[torch.Tensor] = None, workspace=None, stream=None):
    """Device path of ``bplx_pointwise_loglik``: posterior arrays ``[S, T]`` float32 and observed matches (the fixture
    index tensors of ``score_grid`` plus ``home_goals`` / ``away_goals`` uint8) on the GPU.

    ``ll[s, m] = log Pois(yh; lh) + log Pois(ya; la) + log tau(yh, ya; lh, la, corr_coef_s)`` with the rates of the
    predict path (neutral venues and confederations included, no clip of the rates), tau clamped at 0 (a match can give
    -inf) and no match weights.  Returns ``(loglik, stats)``: ``loglik`` is the match-major ``[M, S]`` float32 matrix
    (a view of the ``[M, ld]`` buffer when one is passed in) or ``None`` when ``want_matrix`` is false; ``stats`` is
    ``[M, 4]`` float64 = (max ll, sum exp(ll - max), sum ll, sum ll^2) over the draws (``compare.waic_from_stats``)."""
    lib = _abi.lib()
    keep = []
    ptr = _device_ptr_fn(keep)
    _check_inputs(samples, observations, ("home_goals", "away_goals"))
    s = _samples_struct(model, samples, ptr)
    o = _observations_struct(observations, ptr)
    M, S = o.fixtures.num_fixtures, s.num_samples
    dev = samples["attack"].device
    workspace = _workspace(workspace, int(lib.bplx_pointwise_loglik_workspace_bytes(C.byref(s), C.byref(o))), dev)
    loglik, ld = _output_matrix(loglik, M, S, dev, want_matrix)
    stats = torch.empty((M, 4), dtype=torch.float64, device=dev)
    _abi.check(lib.bplx_pointwise_loglik(C.byref(s), C.byref(o), _dptr(loglik), ld, _dptr(stats), _dptr(workspace),
                                         workspace.numel(), _stream_ptr(stream)))
    return (loglik[:M, :S] if want_matrix else None), stats


def psis_loo(loglik: torch.Tensor, r_eff: float = 1.0, stream=None):
    """Device path of ``bplx_psis_loo``: PSIS-LOO (ArviZ's ``_psislw`` / ``_gpdfit``) per row of the match-major
    ``[M, S]`` float32 matrix (unit inner stride; the row pitch is passed as the leading dimension).  Returns
    ``(elpd_i [M], pareto_k [M])`` float64 on the device: ``elpd_i[m] = logsumexp_s(lw + ll)`` with the Pareto-smoothed
    normalised log-weights ``lw`` of the ratios ``-ll[m]``, ``pareto_k[m]`` the fitted shape (+inf when the tail has at
    most 4 draws).  A row with a non-finite entry gives (NaN, +inf).  The tail, ``ceil(min(0.2 S, 3 sqrt(S / r_eff)))``
    draws, must not exceed ``_abi.PSIS_MAX_TAIL``."""
    assert loglik.is_cuda and loglik.dtype == torch.float32 and loglik.dim() == 2
    assert loglik.stride(1) == 1 or loglik.shape[1] == 1
    lib = _abi.lib()
    M, S = int(loglik.shape[0]), int(loglik.shape[1])
    ld = int(loglik.stride(0)) if M > 1 else S
    elpd = torch.empty(M, dtype=torch.float64, device=loglik.device)
    khat = torch.empty(M, dtype=torch.float64, device=loglik.device)
    _abi.check(lib.bplx_psis_loo(_dptr(loglik), M, S, ld, C.c_double(r_eff), _dptr(elpd), _dptr(khat), None, 0,
                                 _stream_ptr(stream)))
    return elpd, khat


def market_names(total_lines=(), margin_lines=()):
    """Names of the rows ``market_draws`` computes per fixture, in its order."""
    names = ["home_win", "draw", "away_win", "both_teams_score", "home_rate", "away_rate"]
    for x in total_lines:
        names += [f"total_over_{float(x):g}", f"total_under_{float(x):g}"]
    for x in margin_lines:
        names += [f"home_margin_over_{float(x):g}", f"home_margin_under_{float(x):g}"]
    return names


def _market_lines(total_lines, margin_lines):
    ln = _abi.MarketLines()
    ln.num_total_lines, ln.num_margin_lines = len(total_lines), len(margin_lines)
    if max(ln.num_total_lines, ln.num_margin_lines) > _abi.MARKET_MAX_LINES:
        raise ValueError(f"at most {_abi.MARKET_MAX_LINES} lines of each kind")
    for i, x in enumerate(total_lines):
        ln.total_lines[i] = float(x)
    for i, x in enumerate(margin_lines):
        ln.margin_lines[i] = float(x)
    return ln


def market_draws(model: str, samples: Dict[str, torch.Tensor], fixtures: Dict[str, torch.Tensor], max_goals: int,
                 total_lines=(), margin_lines=(), want_matrix: bool = True, draws: Optional[torch.Tensor] = None,
                 workspace=None, stream=None):
    """Device path of ``bplx_market_draws``: per posterior draw and fixture, the K rows of ``market_names(total_lines,
    margin_lines)`` read off the draw's own (unnormalised) score grid up to ``max_goals`` (include/bplx.h gives the
    definitions).  ``samples`` / ``fixtures`` as for ``score_grid``.  Returns ``(draws, stats, invalid)``: ``draws`` the
    row-major ``[F K, S]`` float32 matrix (row ``f K + r``; a view of the ``[F K, ld]`` buffer when one is passed in) or
    None when ``want_matrix`` is false, ``stats [F K, 2]`` float64 (mean and sd over the draws, the same bits with or
    without the matrix and whichever fixtures share the call), ``invalid`` (int32 ``[1]``: (draw, fixture) pairs with a
    non-finite rate)."""
    lib = _abi.lib()
    keep = []
    ptr = _device_ptr_fn(keep)
    _check_inputs(samples, fixtures)
    s = _samples_struct(model, samples, ptr)
    f = _fixtures_struct(fixtures, ptr)
    ln = _market_lines(total_lines, margin_lines)
    F, S, K = f.num_fixtures, s.num_samples, 6 + 2 * len(total_lines) + 2 * len(margin_lines)
    dev = samples["attack"].device
    need = int(lib.bplx_market_draws_workspace_bytes(C.byref(s), C.byref(f), int(max_goals), C.byref(ln)))
    workspace = _workspace(workspace, need, dev)
    draws, ld = _output_matrix(draws, F * K, S, dev, want_matrix)
    stats = torch.empty((F * K, 2), dtype=torch.float64, device=dev)
    invalid = torch.empty(1, dtype=torch.int32, device=dev)
    _abi.check(lib.bplx_market_draws(C.byref(s), C.byref(f), int(max_goals), C.byref(ln), _dptr(draws), ld,
                                     _dptr(stats), _dptr(invalid), _dptr(workspace), workspace.numel(),
                                     _stream_ptr(stream)))
    return (draws[:F * K, :S] if want_matrix else None), stats, invalid


def row_quantiles(rows: torch.Tensor, levels=(), odds: Optional[torch.Tensor] = None, stream=None):
    """Device path of ``bplx_row_quantiles`` over the ``[R, S]`` float32 matrix ``rows`` (unit inner stride; the row
    pitch is passed as the leading dimension): ``quantiles [R, len(levels)]`` float64, numpy's ``method="linear"`` on
    each row's values with exact order statistics, and with ``odds`` (float64 ``[R]`` on the device; <= 0 = none)
    ``exceed [R]`` int64, the number of values v with ``v * odds > 1`` in float64 (else None)."""
    assert rows.is_cuda and rows.dtype == torch.float32 and rows.dim() == 2
    assert rows.stride(1) == 1 or rows.shape[1] == 1
    lib = _abi.lib()
    R, S = int(rows.shape[0]), int(rows.shape[1])
    ld = int(rows.stride(0)) if R > 1 else S
    lv = np.ascontiguousarray(levels, dtype=np.float64).ravel()
    quantiles = torch.empty((R, len(lv)), dtype=torch.float64, device=rows.device)
    exceed = None
    if odds is not None:
        assert odds.is_cuda and odds.dtype == torch.float64 and odds.is_contiguous() and odds.numel() == R
        exceed = torch.empty(R, dtype=torch.int64, device=rows.device)
    _abi.check(lib.bplx_row_quantiles(_dptr(rows), R, S, ld, lv.ctypes.data if len(lv) else None, len(lv),
                                      _dptr(odds), _dptr(quantiles) if len(lv) else None, _dptr(exceed),
                                      _stream_ptr(stream)))
    return quantiles, exceed


_TABLE_ARRAYS = ("start_points", "start_goals_for", "start_goals_against")


def simulate_table(model: str, samples: Dict[str, torch.Tensor], fixtures: Dict[str, torch.Tensor], table: dict,
                   max_goals: int, sims_per_draw: int, seed: int, first_draw: int = 0, want_positions: bool = False,
                   want_scores: bool = False, workspace=None, stream=None,
                   conditions: Optional[dict] = None) -> Dict[str, Optional[torch.Tensor]]:
    """Device path of ``bplx_simulate_table``: season / group-stage simulation, one posterior draw per simulated season.

    ``samples``: posterior arrays ``[S, T]`` on the GPU (the draws of this call; ``first_draw`` is the global index of
    the first one).  ``fixtures``: the index tensors of ``score_grid`` plus ``home_slot`` / ``away_slot`` (uint8 table
    slots).  ``table``: ``start_points``, ``start_goals_for``, ``start_goals_against`` (int32 ``[T_tab]``), ``group``
    (uint8 ``[T_tab]`` or None) on the GPU, and the ints ``num_positions`` (largest group), ``num_points_bins``,
    ``points_win``, ``points_draw`` (``season.build_table`` / ``season.fixture_slots`` make them), and optionally
    ``tiebreak`` (``"goal_difference"``, the default, or ``"head_to_head"``) with the host ``played_h2h`` (int32 ``[T_tab,
    T_tab, 2]``: points and goals of slot u against slot v in played matches, or None).

    Simulation ``n = (first_draw + s) R + r`` uses draw s and the Philox words of ``curand_init(seed, n, 0)``: words 2f,
    2f+1 sample fixture f's score from the draw's own grid (tau clamped at 0, normalised by its sum), word 2F + t is slot
    t's tie-break key.  Teams are ranked within their group by points, then under ``"goal_difference"`` by goal
    difference, goals for, then the key (``bplx_simulate_table``); under ``"head_to_head"`` by the points, goal
    difference and goals for of the matches among the teams level on points (played and simulated), reapplied to the
    teams still level, then overall goal difference, goals for and the key (``bplx_simulate_table_ex``: the same Philox
    words, only the group order can differ).  Fair-play rules are not modelled: ties left are decided by lot.  Returns
    ``position_counts [T_tab, P]`` and ``points_counts [T_tab, B]`` (points gained; int64), ``invalid`` (int64 ``[1]``:
    simulations with a non-finite rate or normaliser, left out of the counts), and when asked ``positions [N, T_tab]``
    and ``scores [N, F, 2]`` (uint8; 255 marks an invalid simulation / fixture), N = S R.

    ``conditions`` (``bplx_simulate_table_conditional``; ``season.build_conditions`` makes it): host arrays
    ``key_fixture`` (int32 ``[Kc]``, strictly increasing fixture indices, 1 <= Kc <= 64), ``event_slot`` (uint8
    ``[E]``) and ``event_positions`` (uint64 ``[E]``: bit p = position p within the slot's group, 1 <= E <= 64).  Key
    fixture j has outcome o in {0 home win, 1 draw, 2 away win} from its sampled score; event e holds iff slot
    ``event_slot[e]``'s position is a bit of ``event_positions[e]``.  Adds ``outcome_counts`` (int64 ``[Kc, 3]``: valid
    simulations in which key fixture j ended in o) and ``conditional_counts`` (int64 ``[Kc, 3, E]``: ... and event e
    held).  No random word is added or moved: every other output is the same bits as without ``conditions``."""
    return _simulate(model, samples, fixtures, table, None, max_goals, sims_per_draw, seed, first_draw, want_positions,
                     want_scores, False, workspace, stream, conditions)


def _table_struct(table: dict, ptr):
    """``_abi.Table`` over the device arrays of ``table``: one slot per entry of ``start_points``."""
    t = _abi.Table()
    t.num_slots = int(table["start_points"].shape[0])
    t.num_positions, t.num_points_bins = int(table["num_positions"]), int(table["num_points_bins"])
    t.points_win, t.points_draw = int(table["points_win"]), int(table["points_draw"])
    t.group = None if table.get("group") is None else ptr(table["group"])
    for k in _TABLE_ARRAYS:
        setattr(t, k, ptr(table[k]))
    return t


def _ranking_struct(table: dict, T_tab: int, keep: list):
    """``_abi.Ranking`` of ``table["tiebreak"]`` over a host copy of ``played_h2h`` (kept alive in ``keep``), or None
    for ``"goal_difference"`` (the calls without a ranking)."""
    rule = table.get("tiebreak", "goal_difference")
    if rule not in TIEBREAKS:
        raise ValueError(f"unknown tiebreak {rule!r} (one of {sorted(TIEBREAKS)})")
    if TIEBREAKS[rule] == _abi.RANK_GOAL_DIFF:
        return None
    r = _abi.Ranking()
    r.rule = TIEBREAKS[rule]
    h2h = table.get("played_h2h")
    if h2h is not None:
        h2h = np.ascontiguousarray(h2h, dtype=np.int32)
        if h2h.shape != (T_tab, T_tab, 2):
            raise ValueError(f"played_h2h has shape {h2h.shape}; the table needs ({T_tab}, {T_tab}, 2)")
        keep.append(h2h)
        r.played_h2h = h2h.ctypes.data
    return r


def _bracket_struct(bracket: dict, keep: list):
    """``_abi.Bracket`` over host copies of the arrays of ``bracket`` (kept alive in ``keep``)."""
    def host(k, dt):
        v = bracket.get(k)
        if v is None:
            return None
        a = np.ascontiguousarray(v, dtype=dt)
        keep.append(a)
        return a.ctypes.data

    b = _abi.Bracket()
    b.num_ties, b.num_rounds = int(len(bracket["round"])), int(bracket["num_rounds"])
    b.num_groups, b.best_position, b.best_count = (int(bracket[k]) for k in ("num_groups", "best_position", "best_count"))
    for k in ("kind", "arg0", "arg1", "round", "neutral_venue", "slot_conf", "best_alloc"):
        setattr(b, k, host(k, np.uint8))
    b.slot_team = host("slot_team", np.uint16)
    return b


def _pairings_struct(bracket: dict, T_tab: int, keep: list):
    """``_abi.Pairings`` over host copies of the pairing arrays of ``bracket`` (kept alive in ``keep``), or None for a
    bracket without pairings."""
    if bracket.get("pool_kind") is None:
        return None

    def host(k, shape=None):
        v = bracket.get(k)
        if v is None:
            return None
        a = np.ascontiguousarray(v, dtype=np.uint8)
        if shape is not None and a.shape != shape:
            raise ValueError(f"{k} has shape {a.shape}; expected {shape}")
        keep.append(a)
        return a.ctypes.data

    P = int(len(bracket["pool_size"]))
    p = _abi.Pairings()
    p.num_pairings = P
    for k in ("mode", "protect", "host_pot"):
        setattr(p, k, host("pairing_" + k, (P,)))
    p.pool_size = host("pool_size", (P,))
    for k in ("pool_kind", "pool_arg0", "pool_arg1", "pool_pot"):
        setattr(p, k, host(k, (P, _abi.PAIRING_MAX_POOL)))
    p.slot_assoc = host("slot_assoc", (T_tab,))
    return p


def simulate_tournament(model: str, samples: Dict[str, torch.Tensor], fixtures: Dict[str, torch.Tensor], table: dict,
                        bracket: dict, max_goals: int, sims_per_draw: int, seed: int, first_draw: int = 0,
                        want_positions: bool = False, want_scores: bool = False, want_knockout: bool = False,
                        workspace=None, stream=None) -> Dict[str, Optional[torch.Tensor]]:
    """Device path of ``bplx_simulate_tournament``: the group stage of ``simulate_table`` (same Philox words, same
    ranking: with the same seed its outputs are bit-identical), then a knockout bracket, one posterior draw per
    simulated tournament.

    ``samples``, ``fixtures``, ``table``: as ``simulate_table`` (``fixtures`` may have no fixtures: a bracket whose
    entrants are all known).  ``bracket``: host arrays ``kind``, ``arg0``, ``arg1`` (uint8 ``[K, 2]``, home and away
    entrant: ``_abi.ENTRANT_*`` and their arguments), ``round`` (``[K]``), ``neutral_venue`` (``[K]`` or None),
    ``slot_team`` (uint16 ``[T_tab]``), ``slot_conf`` (``[T_tab]``, NeutralWC), ``best_alloc`` (``[2^num_groups,
    best_count]`` or None) and the ints ``num_rounds``, ``num_groups``, ``best_position``, ``best_count``
    (``season.build_bracket`` makes them).

    Tie k uses words 2F + T_tab + 3k and + 1 for its score, from the draw's own grid like a group fixture, and + 2 for
    the decider of a drawn tie: the home entrant goes through iff ``u_d (hw_s + aw_s) <= hw_s`` with ``hw_s`` / ``aw_s``
    the draw's own home / away win masses, i.e. with probability ``hw_s / (hw_s + aw_s)`` per draw (the per-draw form of
    ``predict_outcome_proba(knockout=True)``, which renormalises after averaging over the draws).  Extra time and
    penalties are not modelled in that format, ``_abi.TIE_ONE_MATCH``, the default.  ``bracket["tie_format"]`` (uint8
    ``[K]``, optional) sets a format per tie: ``TIE_ONE_MATCH_ET`` (a drawn match goes to extra time, then penalties)
    or ``TIE_TWO_LEGS`` (the away entrant B hosts leg 2 with the venues swapped; level on aggregate: extra time in leg
    2, then penalties; no away-goals rule; never at a neutral venue).  Extra time is played at the venue of the last
    match with the draw's rates times ``EXTRA_TIME_FRACTION`` = 1/3 and no tau correction; the home entrant A wins a
    shoot-out iff ``u_d <= 1/2``.  Tie k's leg 2 and extra time use the Philox block ``E/4 + k``, ``E = 4 ceil((2F +
    T_tab + 3K) / 4)`` (every word at a fixed address: a bracket of format-0 ties gives ``bplx_simulate_tournament``'s
    outputs bit for bit).  Returns ``simulate_table``'s outputs plus ``reach_counts`` / ``win_counts`` (int64 ``[T_tab,
    num_rounds]``: ties of round r the slot played / won; a two-legged tie counts once), ``decided_counts`` (int64
    ``[K, 3]``: tie k settled in normal time or on aggregate / in extra time / by ``u_d``), and when ``want_knockout``
    ``ko_entrants``, ``ko_scores`` (uint8 ``[N, K, 2]``, the first or only match), ``ko_winners`` (``[N, K]``) and
    ``ko_extra`` (``[N, K, 4]``: leg-2 goals of A and B, then extra-time goals of A and B; 254 where not played); 255
    marks an invalid simulation.  ``table["tiebreak"]`` ranks the groups as in ``simulate_table``
    (``bplx_simulate_tournament_ranked``); best-placed qualifiers are ranked across groups by points, goal difference,
    goals for, then the key under either rule.

    Pairings drawn by lot (``bplx_simulate_tournament_paired``): ``bracket`` may also hold ``pairing_mode``,
    ``pairing_protect``, ``pairing_host_pot``, ``pool_size`` (uint8 ``[P]``), ``pool_kind``, ``pool_arg0``,
    ``pool_arg1``, ``pool_pot`` (``[P, 64]``) and ``slot_assoc`` (``[T_tab]`` or None), as ``season.build_bracket``
    makes them; a tie then takes both sides from pair i of pairing d (``_abi.ENTRANT_PAIRED``, arg0 d, arg1 2i and 2i + 1).
    Pairing d is made when its first tie is reached, on the Philox words of blocks ``E/4 + K + 16 d`` onwards: an open
    draw shuffles the pool (``j = i + ((w_i (n - i)) >> 32)``, swap; pair i = the entrants drawn 2i and 2i + 1, the first
    at home); a seeded draw takes an unseeded entrant b (``(w_2i |B left|) >> 32``), then one of the seeded entrants
    left that b may meet (group / association protection) for which the rest can still be paired (``(w_2i+1
    |eligible|) >> 32``), in pool order.  A pool that cannot be paired makes the simulation invalid.  Adds
    ``pairing_counts`` (int64 ``[P, T_tab, T_tab]``: pairing d drew slot u at home against slot v).  A bracket
    without pairings takes ``bplx_simulate_tournament_ranked``'s path and words."""
    return _simulate(model, samples, fixtures, table, bracket, max_goals, sims_per_draw, seed, first_draw,
                     want_positions, want_scores, want_knockout, workspace, stream)


def _conditions_struct(conditions: dict, keep: list):
    """``_abi.Conditions`` over host copies of the arrays of ``conditions`` (kept alive in ``keep``)."""
    arrays = {k: np.ascontiguousarray(conditions[k], dtype=dt).ravel()
              for k, dt in (("key_fixture", np.int32), ("event_slot", np.uint8), ("event_positions", np.uint64))}
    if len(arrays["event_slot"]) != len(arrays["event_positions"]):
        raise ValueError("event_slot and event_positions differ in length")
    keep.extend(arrays.values())
    c = _abi.Conditions()
    c.num_key_fixtures, c.num_events = len(arrays["key_fixture"]), len(arrays["event_slot"])
    for k, a in arrays.items():
        setattr(c, k, a.ctypes.data)
    return c


def _simulate(model, samples, fixtures, table, bracket, max_goals, sims_per_draw, seed, first_draw, want_positions,
              want_scores, want_knockout, workspace, stream, conditions=None):
    """``simulate_tournament``, and ``simulate_table`` when ``bracket`` is None (``bplx_simulate_table``: the group
    stage kernel)."""
    lib = _abi.lib()
    keep = []
    ptr = _device_ptr_fn(keep)
    F = int(len(fixtures["home_team"])) if fixtures.get("home_team") is not None else 0
    _check_inputs(samples, fixtures, ("home_slot", "away_slot") if F else ())
    for k in _TABLE_ARRAYS:
        assert table[k].dtype == torch.int32, k
    T_tab = int(table["start_points"].shape[0])
    if T_tab > _abi.SIM_MAX_TEAMS:
        raise ValueError(f"the table has {T_tab} slots; at most {_abi.SIM_MAX_TEAMS} are supported")
    if F:
        top = int(torch.maximum(fixtures["home_slot"].max(), fixtures["away_slot"].max()))
        if top >= T_tab:
            raise ValueError(f"a fixture names table slot {top}, but the table has {T_tab} slots")
    s = _samples_struct(model, samples, ptr)
    f = _fixtures_struct(fixtures, ptr) if F else _abi.Fixtures()
    t = _table_struct(table, ptr)
    b = None if bracket is None else _bracket_struct(bracket, keep)
    r = _ranking_struct(table, T_tab, keep)
    pg = None if b is None else _pairings_struct(bracket, T_tab, keep)
    cd = None if conditions is None else _conditions_struct(conditions, keep)
    structs = (C.byref(s), C.byref(f), C.byref(t)) + (() if b is None else (C.byref(b),))
    if pg is not None:
        need = int(lib.bplx_simulate_tournament_paired_workspace_bytes(*structs, None if r is None else C.byref(r),
                                                                        C.byref(pg)))
    elif r is None:
        ws_bytes = lib.bplx_simulate_workspace_bytes if b is None else lib.bplx_simulate_tournament_workspace_bytes
        need = int(ws_bytes(*structs))
    else:
        ws_bytes = (lib.bplx_simulate_table_ex_workspace_bytes if b is None
                    else lib.bplx_simulate_tournament_ranked_workspace_bytes)
        need = int(ws_bytes(*structs, C.byref(r)))
    dev = samples["attack"].device
    workspace = _workspace(workspace, need, dev)
    N = s.num_samples * int(sims_per_draw)
    i64 = dict(dtype=torch.int64, device=dev)
    u8 = dict(dtype=torch.uint8, device=dev)
    out = {"position_counts": torch.empty((T_tab, t.num_positions), **i64),
           "points_counts": torch.empty((T_tab, t.num_points_bins), **i64)}
    if cd is not None:
        out.update(outcome_counts=torch.empty((cd.num_key_fixtures, 3), **i64),
                   conditional_counts=torch.empty((cd.num_key_fixtures, 3, cd.num_events), **i64))
    if b is not None:
        out.update(reach_counts=torch.empty((T_tab, b.num_rounds), **i64),
                   win_counts=torch.empty((T_tab, b.num_rounds), **i64),
                   decided_counts=torch.empty((b.num_ties, 3), **i64))
        if pg is not None:
            out["pairing_counts"] = torch.empty((pg.num_pairings, T_tab, T_tab), **i64)
    out.update(invalid=torch.empty(1, **i64), positions=torch.empty((N, T_tab), **u8) if want_positions else None,
               scores=torch.empty((N, F, 2), **u8) if want_scores else None)
    if b is not None:
        K = b.num_ties
        out.update(ko_entrants=torch.empty((N, K, 2), **u8) if want_knockout else None,
                   ko_scores=torch.empty((N, K, 2), **u8) if want_knockout else None,
                   ko_winners=torch.empty((N, K), **u8) if want_knockout else None,
                   ko_extra=torch.empty((N, K, 4), **u8) if want_knockout else None)
    # the C functions take the outputs in the order of `out`, with `invalid` last
    outputs = [_dptr(v) for k, v in out.items() if k != "invalid"] + [_dptr(out["invalid"])]
    slots = (ptr(fixtures["home_slot"]), ptr(fixtures["away_slot"])) if F else (None, None)
    if b is None:
        run, args = lib.bplx_simulate_table, structs[:2] + slots + structs[2:]
        if cd is not None:
            run, args = lib.bplx_simulate_table_conditional, args + (None if r is None else C.byref(r), C.byref(cd))
        elif r is not None:
            run, args = lib.bplx_simulate_table_ex, args + (C.byref(r),)
    else:
        fmt = bracket.get("tie_format")
        if fmt is not None:
            fmt = np.ascontiguousarray(fmt, dtype=np.uint8)
            if fmt.shape != (b.num_ties,):
                raise ValueError(f"tie_format has shape {fmt.shape}; the bracket has {b.num_ties} ties")
            keep.append(fmt)
        run, args = lib.bplx_simulate_tournament_ex, structs[:2] + slots + structs[2:] + (
            None if fmt is None else fmt.ctypes.data,)
        if pg is not None:
            run, args = lib.bplx_simulate_tournament_paired, args + (None if r is None else C.byref(r), C.byref(pg))
        elif r is not None:
            run, args = lib.bplx_simulate_tournament_ranked, args + (C.byref(r),)
    _abi.check(run(*args, int(max_goals), int(sims_per_draw), _seed(seed), int(first_draw),
                   *outputs, _dptr(workspace), workspace.numel(), _stream_ptr(stream)))
    return out



def posterior_predictive(model: str, samples: Dict[str, torch.Tensor], observations: Dict[str, torch.Tensor],
                         max_goals: int = 15, score_bins: int = 6, points=(3, 1), sims_per_draw: int = 1, seed: int = 0,
                         first_draw: int = 0, want_scores: bool = False, workspace=None,
                         stream=None) -> Dict[str, Optional[torch.Tensor]]:
    """Device path of ``bplx_posterior_predictive``: replicated datasets of the observed matches, one posterior draw per
    replicate, each reduced to its statistics on the GPU.

    ``samples``: posterior arrays ``[S, T]`` on the GPU (the draws of this call; ``first_draw`` is the global index of
    the first one).  ``observations``: the index tensors of ``score_grid`` plus ``home_goals`` / ``away_goals`` (uint8),
    as for ``pointwise_loglik``.

    Replicate ``n = (first_draw + s) R + r`` (R = ``sims_per_draw``) uses draw s; words 2m and 2m + 1 of
    ``curand_init(seed, n, 0)`` sample match m's score with the season simulation's sampler (the draw's own grid up to
    ``max_goals``, tau clamped at 0, normalised by its sum), so with the same seed, draws and matches the scores equal
    ``simulate_table``'s.  Match weights are ignored.  Returns per replicate (row ``s R + r``, N = S R):
    ``score_counts [N, B, B]`` (cells ``min(hg, B-1), min(ag, B-1)``, B = ``score_bins``), ``outcome_counts [N, 3]``
    (home wins, draws, away wins), ``team_points``, ``team_goals_for``, ``team_goals_against [N, T]`` (int32),
    ``goals [N, 2]`` (home, away) and ``total_goals_sq [N]`` (sum of squared match totals; int64); ``invalid`` (int64
    ``[1]``: replicates with a non-finite rate or normaliser, whose rows are -1), and when ``want_scores`` the raw
    ``scores [N, M, 2]`` (uint8; 255 marks the match that made a replicate invalid)."""
    lib = _abi.lib()
    keep = []
    ptr = _device_ptr_fn(keep)
    _check_inputs(samples, observations, ("home_goals", "away_goals"))
    s = _samples_struct(model, samples, ptr)
    o = _observations_struct(observations, ptr)
    B = int(score_bins)
    dev = samples["attack"].device
    workspace = _workspace(workspace, int(lib.bplx_posterior_predictive_workspace_bytes(C.byref(s), C.byref(o))), dev)
    res, out = _ppc_outputs(s.num_samples * int(sims_per_draw), o.fixtures.num_fixtures, s.num_teams, B, dev,
                            want_scores)
    pw, pd = (int(x) for x in points)
    _abi.check(lib.bplx_posterior_predictive(C.byref(s), C.byref(o), int(max_goals), B, pw, pd, int(sims_per_draw),
                                             _seed(seed), int(first_draw), C.byref(out), _dptr(workspace),
                                             workspace.numel(), _stream_ptr(stream)))
    return res


# ---- the dynamic model's predictive distribution ----------------------------------------------------------------
_FORECAST_SITES = ("attack", "defence", "home_attack", "away_attack", "home_defence", "away_defence")


def dynamic_forecast(attack_last: torch.Tensor, defence_last: torch.Tensor, horizon: int, seed: int,
                     first_draw: int = 0, stream=None) -> Dict[str, torch.Tensor]:
    """Device path of ``bplx_dynamic_forecast``: the dynamic model's gameweeks ``G .. G + horizon - 1`` drawn from its
    own generative process, continued from the walk at gameweek ``G - 1`` (``attack_last`` / ``defence_last [S, T]``
    float32 on the GPU, draws ``first_draw ..``).  Returns the six NEUTRAL sites ``[horizon, S, T]``: ``attack``,
    ``defence``, ``home_attack``, ``away_attack``, ``home_defence``, ``away_defence`` (word map in include/bplx.h)."""
    lib = _abi.lib()
    assert attack_last.is_cuda and attack_last.dtype == torch.float32 and attack_last.is_contiguous()
    assert defence_last.shape == attack_last.shape and defence_last.dtype == torch.float32 and defence_last.is_contiguous()
    S, T = int(attack_last.shape[0]), int(attack_last.shape[1])
    out = {k: torch.empty((int(horizon), S, T), dtype=torch.float32, device=attack_last.device) for k in _FORECAST_SITES}
    _abi.check(lib.bplx_dynamic_forecast(_dptr(attack_last), _dptr(defence_last), S, T, int(horizon),
                                         _seed(seed), int(first_draw), *(_dptr(out[k]) for k in _FORECAST_SITES),
                                         _stream_ptr(stream)))
    return out


def _gameweek_major(samples: Dict[str, torch.Tensor]):
    """``[G', S, T]`` sample arrays (``corr_coef [G', S]``) -> the ``[G' S, ...]`` pseudo-draws the C ABI takes, G', S."""
    G, S = int(samples["attack"].shape[0]), int(samples["attack"].shape[1])
    flat = {k: None if v is None else v.reshape((G * S,) + tuple(v.shape[2:])) for k, v in samples.items()}
    return flat, G, S


def take_rows(v: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """``v[idx]`` along the first axis; uint16 team indices go through their int16 view (torch has no uint16 gather)."""
    if v.dtype == torch.uint16:
        return v.view(torch.int16).index_select(0, idx).view(torch.uint16)
    return v.index_select(0, idx)


def _gw_observations(samples, observations, gameweek, keep):
    ptr = _device_ptr_fn(keep)
    _check_inputs(samples, observations, ("home_goals", "away_goals"))
    o = _observations_struct(observations, ptr)
    gw = np.ascontiguousarray(gameweek, dtype=np.int32)
    keep.append(gw)
    return o, gw


def pointwise_loglik_gameweeks(model: str, samples: Dict[str, torch.Tensor], observations: Dict[str, torch.Tensor],
                               gameweek, want_matrix: bool = True, loglik: Optional[torch.Tensor] = None,
                               workspace=None, stream=None):
    """``pointwise_loglik`` for matches spread over gameweeks, in one launch (``bplx_pointwise_loglik_gameweeks``).
    ``samples``: NEUTRAL-form arrays ``[G', S, T]`` (``corr_coef [G', S]``) on the GPU, gameweek-major; ``gameweek``:
    host ints ``[M]`` in ``[0, G')``, match m's gameweek.  The matches are grouped by gameweek here (a stable sort) and
    the outputs returned in the order given: ``(loglik [M, S] or None, stats [M, 4])``.  ``loglik`` (an ``[M, ld]``
    buffer) is only filled in place when the matches are already grouped."""
    lib = _abi.lib()
    gw = np.asarray(gameweek, dtype=np.int64)
    order = np.argsort(gw, kind="stable")
    grouped = bool((np.diff(gw) >= 0).all())
    if not grouped:
        idx = torch.from_numpy(order).to(observations["home_team"].device)
        observations = {k: take_rows(v, idx) for k, v in observations.items()}
        gw, loglik = gw[order], None
    flat, G, S = _gameweek_major(samples)
    keep = []
    s = _samples_struct(model, flat, _device_ptr_fn(keep))
    o, gw32 = _gw_observations(flat, observations, gw, keep)
    M = o.fixtures.num_fixtures
    dev = samples["attack"].device
    workspace = _workspace(workspace, int(lib.bplx_pointwise_loglik_gameweeks_workspace_bytes(C.byref(s), G,
                                                                                              C.byref(o))), dev)
    loglik, ld = _output_matrix(loglik, M, S, dev, want_matrix)
    stats = torch.empty((M, 4), dtype=torch.float64, device=dev)
    _abi.check(lib.bplx_pointwise_loglik_gameweeks(C.byref(s), G, C.byref(o), gw32.ctypes.data, _dptr(loglik), ld,
                                                   _dptr(stats), _dptr(workspace), workspace.numel(),
                                                   _stream_ptr(stream)))
    ll = loglik[:M, :S] if want_matrix else None
    if not grouped:
        inv = torch.from_numpy(np.argsort(order, kind="stable")).to(dev)
        stats = stats.index_select(0, inv)
        ll = None if ll is None else ll.index_select(0, inv)
    return ll, stats


def posterior_predictive_gameweeks(model: str, samples: Dict[str, torch.Tensor], observations: Dict[str, torch.Tensor],
                                   gameweek, max_goals: int = 15, score_bins: int = 6, points=(3, 1),
                                   sims_per_draw: int = 1, seed: int = 0, first_draw: int = 0,
                                   want_scores: bool = False, workspace=None,
                                   stream=None) -> Dict[str, Optional[torch.Tensor]]:
    """``posterior_predictive`` for matches spread over gameweeks (``bplx_posterior_predictive_gameweeks``):
    ``samples`` NEUTRAL-form ``[G', S, T]`` (``corr_coef [G', S]``) on the GPU, ``gameweek`` host ints ``[M]`` in
    ``[0, G')``; match m of draw s is sampled from gameweek ``gameweek[m]``'s row, with the replicate index, words and
    statistics of ``posterior_predictive`` (matches in the order given).  Same outputs."""
    lib = _abi.lib()
    flat, G, S = _gameweek_major(samples)
    keep = []
    s = _samples_struct(model, flat, _device_ptr_fn(keep))
    o, gw32 = _gw_observations(flat, observations, gameweek, keep)
    B = int(score_bins)
    dev = samples["attack"].device
    workspace = _workspace(workspace, int(lib.bplx_posterior_predictive_gameweeks_workspace_bytes(C.byref(s), G,
                                                                                                  C.byref(o))), dev)
    res, out = _ppc_outputs(S * int(sims_per_draw), o.fixtures.num_fixtures, s.num_teams, B, dev, want_scores)
    pw, pd = (int(x) for x in points)
    _abi.check(lib.bplx_posterior_predictive_gameweeks(C.byref(s), G, C.byref(o), gw32.ctypes.data, int(max_goals), B,
                                                       pw, pd, int(sims_per_draw), _seed(seed), int(first_draw),
                                                       C.byref(out), _dptr(workspace), workspace.numel(),
                                                       _stream_ptr(stream)))
    return res
