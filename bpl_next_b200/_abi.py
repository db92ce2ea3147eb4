"""ctypes binding of ``include/bplx.h`` (the C ABI of ``libbplx.so``).

This is the binding a maintainer of bpl-next would add for this path (INTEGRATION.md shows the
``jax.ffi`` variant); there is no CPU fallback: importing the library raises if the CUDA shared
object has not been built (``python -c "import __graft_entry__ as g; g.build()"``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libbplx.so")

# bplx_status
OK, E_INVALID, E_UNSUPPORTED, E_CUDA, E_NOMEM, E_WORKSPACE = 0, -1, -2, -3, -4, -5
# bplx_model
DIXON_COLES, EXTENDED, NEUTRAL, NEUTRAL_WC, DYNAMIC = 0, 1, 2, 3, 4
MODEL_IDS = {"dixon_coles": 0, "extended": 1, "neutral": 2, "neutral_wc": 3, "dynamic": 4}
# bplx_layout
CHAIN_MAJOR, CHAIN_MINOR = 0, 1


class ProblemDesc(C.Structure):
    _fields_ = [
        ("model", C.c_int32), ("num_matches", C.c_int32), ("num_teams", C.c_int32),
        ("num_covariates", C.c_int32), ("num_conferences", C.c_int32), ("num_gameweeks", C.c_int32),
        ("flags", C.c_uint32),
        ("home_team", C.POINTER(C.c_uint16)), ("away_team", C.POINTER(C.c_uint16)),
        ("home_goals", C.POINTER(C.c_uint8)), ("away_goals", C.POINTER(C.c_uint8)),
        ("neutral_venue", C.POINTER(C.c_uint8)),
        ("home_conf", C.POINTER(C.c_uint8)), ("away_conf", C.POINTER(C.c_uint8)),
        ("gameweek", C.POINTER(C.c_int32)),
        ("weights", C.POINTER(C.c_float)),
        ("covariates", C.POINTER(C.c_float)),
    ]


class Samples(C.Structure):
    _fields_ = [
        ("model", C.c_int32), ("num_samples", C.c_int32), ("num_teams", C.c_int32), ("num_conferences", C.c_int32),
        ("attack", C.c_void_p), ("defence", C.c_void_p),
        ("home_attack", C.c_void_p), ("away_attack", C.c_void_p),
        ("home_defence", C.c_void_p), ("away_defence", C.c_void_p),
        ("confederation_strength", C.c_void_p), ("corr_coef", C.c_void_p),
    ]


class Fixtures(C.Structure):
    _fields_ = [
        ("num_fixtures", C.c_int32),
        ("home_team", C.c_void_p), ("away_team", C.c_void_p),
        ("home_conf", C.c_void_p), ("away_conf", C.c_void_p), ("neutral_venue", C.c_void_p),
    ]


class Observations(C.Structure):
    _fields_ = [("fixtures", Fixtures), ("home_goals", C.c_void_p), ("away_goals", C.c_void_p)]


class Table(C.Structure):
    _fields_ = [
        ("num_slots", C.c_int32), ("num_positions", C.c_int32), ("num_points_bins", C.c_int32),
        ("points_win", C.c_int32), ("points_draw", C.c_int32),
        ("group", C.c_void_p), ("start_points", C.c_void_p), ("start_goals_for", C.c_void_p),
        ("start_goals_against", C.c_void_p),
    ]


class Bracket(C.Structure):
    _fields_ = [
        ("num_ties", C.c_int32), ("num_rounds", C.c_int32), ("num_groups", C.c_int32), ("best_position", C.c_int32),
        ("best_count", C.c_int32),
        ("kind", C.c_void_p), ("arg0", C.c_void_p), ("arg1", C.c_void_p), ("round", C.c_void_p),
        ("neutral_venue", C.c_void_p), ("slot_team", C.c_void_p), ("slot_conf", C.c_void_p), ("best_alloc", C.c_void_p),
    ]


class Ranking(C.Structure):
    _fields_ = [("rule", C.c_int32), ("played_h2h", C.c_void_p)]


class PpcOutput(C.Structure):
    _fields_ = [
        ("score_counts", C.c_void_p), ("outcome_counts", C.c_void_p), ("goals", C.c_void_p),
        ("total_goals_sq", C.c_void_p), ("team_points", C.c_void_p), ("team_goals_for", C.c_void_p),
        ("team_goals_against", C.c_void_p), ("scores", C.c_void_p), ("invalid", C.c_void_p),
    ]


PSIS_MAX_TAIL = 16384  # BPLX_PSIS_MAX_TAIL
SIM_MAX_TEAMS = 64  # BPLX_SIM_MAX_TEAMS
KO_MAX_TIES, KO_MAX_ROUNDS, KO_MAX_BEST, KO_MAX_ALLOC_GROUPS = 64, 16, 16, 16  # BPLX_KO_MAX_*
# BPLX_ENTRANT_*
ENTRANT_SLOT, ENTRANT_GROUP_POS, ENTRANT_BEST, ENTRANT_WINNER, ENTRANT_LOSER = 0, 1, 2, 3, 4
# BPLX_TIE_*, BPLX_EXTRA_TIME_FRACTION
TIE_ONE_MATCH, TIE_ONE_MATCH_ET, TIE_TWO_LEGS = 0, 1, 2
EXTRA_TIME_FRACTION = 1.0 / 3.0
# BPLX_RANK_*
RANK_GOAL_DIFF, RANK_HEAD_TO_HEAD = 0, 1


class BplxError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"bplx status {status}: {message}")
        self.status = status


_lib = None


def declare(lib):
    """Attach argtypes / restypes for every symbol of include/bplx.h."""
    vp, i, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.bplx_problem_create.argtypes = [C.POINTER(ProblemDesc), C.POINTER(vp)]
    lib.bplx_problem_create.restype = i
    lib.bplx_problem_destroy.argtypes = [vp]
    lib.bplx_problem_destroy.restype = None
    lib.bplx_num_params.argtypes = [vp]
    lib.bplx_num_params.restype = i
    lib.bplx_problem_layout.argtypes = [vp]
    lib.bplx_problem_layout.restype = C.c_char_p
    lib.bplx_problem_stats.argtypes = [vp, C.POINTER(C.c_longlong), i]
    lib.bplx_problem_stats.restype = i
    lib.bplx_problem_warp_stats.argtypes = [vp, C.POINTER(C.c_longlong), i]
    lib.bplx_problem_warp_stats.restype = i
    lib.bplx_logdensity_workspace_bytes.argtypes = [vp, i]
    lib.bplx_logdensity_workspace_bytes.restype = sz
    lib.bplx_logdensity_fwdbwd.argtypes = [vp, i, i, i, vp, vp, vp, vp, vp, sz, vp]
    lib.bplx_logdensity_fwdbwd.restype = i
    lib.bplx_loglik_num_inputs.argtypes = [vp]
    lib.bplx_loglik_num_inputs.restype = i
    lib.bplx_loglik_layout.argtypes = [vp]
    lib.bplx_loglik_layout.restype = C.c_char_p
    lib.bplx_loglik_fwdbwd.argtypes = [vp, i, i, i, vp, vp, vp, vp, vp, sz, vp]
    lib.bplx_loglik_fwdbwd.restype = i
    lib.bplx_logdensity_fwdbwd_host.argtypes = [vp, i, vp, vp, vp, vp]
    lib.bplx_logdensity_fwdbwd_host.restype = i
    lib.bplx_score_grid_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), i]
    lib.bplx_score_grid_workspace_bytes.restype = sz
    lib.bplx_score_grid.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), i, C.c_float, vp, vp, vp, sz, vp]
    lib.bplx_score_grid.restype = i
    lib.bplx_score_grid_ex.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), i, C.c_float, vp, vp, vp, sz, vp, C.c_uint]
    lib.bplx_score_grid_ex.restype = i
    lib.bplx_score_grid_host.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), i, C.c_float, vp, vp]
    lib.bplx_score_grid_host.restype = i
    lib.bplx_pointwise_loglik_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Observations)]
    lib.bplx_pointwise_loglik_workspace_bytes.restype = sz
    lib.bplx_pointwise_loglik.argtypes = [C.POINTER(Samples), C.POINTER(Observations), vp, sz, vp, vp, sz, vp]
    lib.bplx_pointwise_loglik.restype = i
    lib.bplx_psis_loo.argtypes = [vp, i, i, sz, C.c_double, vp, vp, vp, sz, vp]
    lib.bplx_psis_loo.restype = i
    lib.bplx_simulate_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), C.POINTER(Table)]
    lib.bplx_simulate_workspace_bytes.restype = sz
    lib.bplx_simulate_table.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), vp, vp, C.POINTER(Table), i, i,
                                        C.c_ulonglong, C.c_longlong, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.bplx_simulate_table.restype = i
    lib.bplx_simulate_tournament_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), C.POINTER(Table),
                                                             C.POINTER(Bracket)]
    lib.bplx_simulate_tournament_workspace_bytes.restype = sz
    lib.bplx_simulate_tournament.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), vp, vp, C.POINTER(Table),
                                             C.POINTER(Bracket), i, i, C.c_ulonglong, C.c_longlong, vp, vp, vp, vp, vp,
                                             vp, vp, vp, vp, vp, vp, sz, vp]
    lib.bplx_simulate_tournament.restype = i
    lib.bplx_simulate_tournament_ex.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), vp, vp, C.POINTER(Table),
                                                C.POINTER(Bracket), vp, i, i, C.c_ulonglong, C.c_longlong, vp, vp, vp,
                                                vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.bplx_simulate_tournament_ex.restype = i
    lib.bplx_simulate_table_ex_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), C.POINTER(Table),
                                                           C.POINTER(Ranking)]
    lib.bplx_simulate_table_ex_workspace_bytes.restype = sz
    lib.bplx_simulate_table_ex.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), vp, vp, C.POINTER(Table),
                                           C.POINTER(Ranking), i, i, C.c_ulonglong, C.c_longlong, vp, vp, vp, vp, vp,
                                           vp, sz, vp]
    lib.bplx_simulate_table_ex.restype = i
    lib.bplx_simulate_tournament_ranked_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures),
                                                                    C.POINTER(Table), C.POINTER(Bracket),
                                                                    C.POINTER(Ranking)]
    lib.bplx_simulate_tournament_ranked_workspace_bytes.restype = sz
    lib.bplx_simulate_tournament_ranked.argtypes = [C.POINTER(Samples), C.POINTER(Fixtures), vp, vp, C.POINTER(Table),
                                                    C.POINTER(Bracket), vp, C.POINTER(Ranking), i, i, C.c_ulonglong,
                                                    C.c_longlong, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                                    sz, vp]
    lib.bplx_simulate_tournament_ranked.restype = i
    lib.bplx_posterior_predictive_workspace_bytes.argtypes = [C.POINTER(Samples), C.POINTER(Observations)]
    lib.bplx_posterior_predictive_workspace_bytes.restype = sz
    lib.bplx_posterior_predictive.argtypes = [C.POINTER(Samples), C.POINTER(Observations), i, i, i, i, i, C.c_ulonglong,
                                              C.c_longlong, C.POINTER(PpcOutput), vp, sz, vp]
    lib.bplx_posterior_predictive.restype = i
    lib.bplx_reload_env.argtypes = []
    lib.bplx_reload_env.restype = None
    lib.bplx_last_error.argtypes = []
    lib.bplx_last_error.restype = C.c_char_p
    lib.bplx_version.argtypes = []
    lib.bplx_version.restype = i
    lib.bplx_peer_sum.argtypes = [C.POINTER(vp), i, i, C.c_size_t, C.c_size_t, C.c_size_t, vp, C.c_size_t, C.c_size_t, vp,
                                  C.c_uint, vp]
    lib.bplx_peer_sum.restype = i
    lib.bplx_launch_count.argtypes = []
    lib.bplx_launch_count.restype = C.c_ulonglong
    return lib


def lib():
    """The loaded shared library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA library first "
                "(`python -c 'import __graft_entry__ as g; g.build()'`). bpl_next_b200 has no CPU fallback."
            )
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(status: int):
    if status != OK:
        raise BplxError(status, lib().bplx_last_error().decode("utf-8", "replace"))
