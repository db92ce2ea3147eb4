"""CPU: the argument checks and workspace sizes of the posterior-draw consumers of the C ABI.

For every consumer with a workspace: the size call returns the recorded number of bytes for a valid shape, and the entry
point given one byte less refuses with BPLX_E_WORKSPACE and names that very number.  Then one-fault mutations of each
shared check (max_goals, points, draw range, observed scores, predictive-check outputs, size-call preconditions,
ranking) must give the recorded status and full error text, or the recorded size.

Every entry call passes workspace = NULL: no call can reach a launch, so the device pointers below are stand-ins that
are never dereferenced.  Arrays the library reads on the host (gameweeks, bracket, pairings, conditions, played_h2h)
are real numpy arrays.  The score grid's plan reads the SM count, 148 without a device as on a B200.
"""
import ctypes as C

import numpy as np
import pytest

from bpl_next_b200 import _abi

S, T, CF, F, NGW = 1000, 20, 4, 38, 4
NT_CUP, F_CUP = 16, 24


def fake(k):
    return 0x7F0000000000 + 0x100000 * k


def ref(x):
    return None if x is None else C.byref(x)


def _struct(cls, o, name, **fields):
    """``cls(**fields)`` with the overrides ``o["name.field"]``; None when ``o[name]`` is None."""
    if name in o and o[name] is None:
        return None
    x = cls(**fields)
    for k, v in o.items():
        if k.startswith(name + "."):
            setattr(x, k[len(name) + 1:], v)
    return x


def _samples(o, num_samples=S):
    ptrs = {k: fake(i) for i, k in enumerate(("attack", "defence", "home_attack", "away_attack", "home_defence",
                                               "away_defence", "confederation_strength", "corr_coef"))}
    return _struct(_abi.Samples, o, "s", model=_abi.NEUTRAL_WC, num_samples=num_samples, num_teams=T,
                   num_conferences=CF, **ptrs)


def _fixtures(o, num_fixtures=F):
    ptrs = {k: fake(10 + i) for i, k in enumerate(("home_team", "away_team", "home_conf", "away_conf",
                                                   "neutral_venue"))}
    return _struct(_abi.Fixtures, o, "f", num_fixtures=num_fixtures, **ptrs)


def _observations(o):
    if "obs" in o and o["obs"] is None:
        return None
    return _struct(_abi.Observations, o, "obs", fixtures=_fixtures(o), home_goals=fake(20), away_goals=fake(21))


def _table(o, slots):
    return _struct(_abi.Table, o, "t", num_slots=slots, num_positions=slots if slots == T else 4,
                   num_points_bins=3 * 2 * F + 1, points_win=3, points_draw=1, group=fake(30), start_points=fake(31),
                   start_goals_for=fake(32), start_goals_against=fake(33))


def _ranking(o, slots, keep):
    played = np.zeros((slots, slots, 2), dtype=np.int32)
    keep.append(played)
    return _struct(_abi.Ranking, o, "r", rule=_abi.RANK_HEAD_TO_HEAD, played_h2h=played.ctypes.data)


def _host(keep, a, dtype):
    a = np.ascontiguousarray(a, dtype=dtype)
    keep.append(a)
    return a.ctypes.data


def _bracket(o, keep, paired):
    """Four groups of four, the group winners and two best third-placed teams (allocation table) in the quarter-finals
    -- or, ``paired``, the first two quarter-finals drawn by lot from the four runners-up."""
    gp, best, win, pr = _abi.ENTRANT_GROUP_POS, _abi.ENTRANT_BEST, _abi.ENTRANT_WINNER, _abi.ENTRANT_PAIRED
    ties = [((gp, 0, 0), (best, 0, 0)), ((gp, 1, 0), (best, 1, 0)), ((gp, 2, 0), (gp, 3, 1)), ((gp, 3, 0), (gp, 2, 1)),
            ((win, 0, 0), (win, 1, 0)), ((win, 2, 0), (win, 3, 0)), ((win, 4, 0), (win, 5, 0))]
    if paired:
        ties[0], ties[1] = ((pr, 0, 0), (pr, 0, 1)), ((pr, 0, 2), (pr, 0, 3))
    e = np.array(ties, dtype=np.uint8)  # [K, 2 sides, (kind, arg0, arg1)]
    return _struct(_abi.Bracket, o, "b", num_ties=len(ties), num_rounds=3, num_groups=4, best_position=2, best_count=2,
                   kind=_host(keep, e[:, :, 0], np.uint8), arg0=_host(keep, e[:, :, 1], np.uint8),
                   arg1=_host(keep, e[:, :, 2], np.uint8), round=_host(keep, [0, 0, 0, 0, 1, 1, 2], np.uint8),
                   neutral_venue=None, slot_team=_host(keep, np.arange(NT_CUP), np.uint16),
                   slot_conf=_host(keep, np.arange(NT_CUP) % CF, np.uint8),
                   best_alloc=_host(keep, np.full((16, 2), 0xFF), np.uint8))


def _pairings(o, keep):
    pool = np.zeros((1, _abi.PAIRING_MAX_POOL), dtype=np.uint8)
    kind, arg0, arg1 = pool.copy(), pool.copy(), pool.copy()
    kind[0, :4], arg0[0, :4], arg1[0, :4] = _abi.ENTRANT_GROUP_POS, np.arange(4), 1
    return _struct(_abi.Pairings, o, "p", num_pairings=1, mode=_host(keep, [_abi.PAIRING_OPEN], np.uint8),
                   protect=None, host_pot=None, pool_size=_host(keep, [4], np.uint8), pool_kind=_host(keep, kind, np.uint8),
                   pool_arg0=_host(keep, arg0, np.uint8), pool_arg1=_host(keep, arg1, np.uint8), pool_pot=None,
                   slot_assoc=None)


def _draw_args(o):
    return (o.get("max_goals", 10), o.get("R", 2), C.c_ulonglong(7), o.get("first_draw", 5))


# ---- the consumers: each returns (size call, entry call taking workspace_bytes), workspace NULL ------------------
def score_grid(o, keep):
    s, f, g = _samples(o), _fixtures(o), o.get("max_goals", 10)
    return (lambda: lib().bplx_score_grid_workspace_bytes(ref(s), ref(f), g),
            lambda n: lib().bplx_score_grid_ex(ref(s), ref(f), g, C.c_float(1.0 / S), fake(40), fake(41), None, n,
                                               None, 0))


def pointwise(o, keep):
    s, obs = _samples(o), _observations(o)
    return (lambda: lib().bplx_pointwise_loglik_workspace_bytes(ref(s), ref(obs)),
            lambda n: lib().bplx_pointwise_loglik(ref(s), ref(obs), fake(40), S, fake(41), None, n, None))


def _gameweeks(o, keep):
    return _host(keep, o.get("gameweek", np.arange(F) * NGW // F), np.int32)


def pointwise_gameweeks(o, keep):
    s, obs, gw, ngw = _samples(o), _observations(o), _gameweeks(o, keep), o.get("ngw", NGW)
    return (lambda: lib().bplx_pointwise_loglik_gameweeks_workspace_bytes(ref(s), ngw, ref(obs)),
            lambda n: lib().bplx_pointwise_loglik_gameweeks(ref(s), ngw, ref(obs), gw, fake(40), S // NGW, fake(41),
                                                            None, n, None))


def markets(o, keep):
    s, f, g = _samples(o), _fixtures(o), o.get("max_goals", 10)
    ln = _struct(_abi.MarketLines, o, "lines", num_total_lines=2, num_margin_lines=1)
    if ln is not None:
        ln.total_lines[0], ln.total_lines[1], ln.margin_lines[0] = 2.5, 3.5, -1.5
    return (lambda: lib().bplx_market_draws_workspace_bytes(ref(s), ref(f), g, ref(ln)),
            lambda n: lib().bplx_market_draws(ref(s), ref(f), g, ref(ln), fake(40), S, fake(41), fake(42), None, n,
                                              None))


def table(o, keep):
    s, f, t = _samples(o), _fixtures(o), _table(o, T)
    return (lambda: lib().bplx_simulate_workspace_bytes(ref(s), ref(f), ref(t)),
            lambda n: lib().bplx_simulate_table(ref(s), ref(f), fake(50), fake(51), ref(t), *_draw_args(o), fake(52),
                                                fake(53), None, None, fake(54), None, n, None))


def table_conditional(o, keep):
    s, f, t, r = _samples(o), _fixtures(o), _table(o, T), _ranking(o, T, keep)
    c = _abi.Conditions(num_key_fixtures=2, key_fixture=_host(keep, [3, 9], np.int32), num_events=2,
                        event_slot=_host(keep, [0, 5], np.uint8), event_positions=_host(keep, [1, 6], np.uint64))
    return (lambda: lib().bplx_simulate_table_ex_workspace_bytes(ref(s), ref(f), ref(t), ref(r)),
            lambda n: lib().bplx_simulate_table_conditional(ref(s), ref(f), fake(50), fake(51), ref(t), ref(r), ref(c),
                                                            *_draw_args(o), fake(52), fake(53), fake(55), fake(56),
                                                            None, None, fake(54), None, n, None))


def _tournament_outputs():
    return (fake(52), fake(53), fake(57), fake(58), fake(59))  # position, points, reach, win, decided counts


def tournament_ranked(o, keep):
    s, f, t, b, r = _samples(o), _fixtures(o, F_CUP), _table(o, NT_CUP), _bracket(o, keep, False), _ranking(o, NT_CUP, keep)
    return (lambda: lib().bplx_simulate_tournament_ranked_workspace_bytes(ref(s), ref(f), ref(t), ref(b), ref(r)),
            lambda n: lib().bplx_simulate_tournament_ranked(ref(s), ref(f), fake(50), fake(51), ref(t), ref(b), None,
                                                            ref(r), *_draw_args(o), *_tournament_outputs(), None, None,
                                                            None, None, None, None, fake(54), None, n, None))


def tournament_paired(o, keep):
    s, f, t, b, r = _samples(o), _fixtures(o, F_CUP), _table(o, NT_CUP), _bracket(o, keep, True), _ranking(o, NT_CUP, keep)
    p = _pairings(o, keep)
    return (lambda: lib().bplx_simulate_tournament_paired_workspace_bytes(ref(s), ref(f), ref(t), ref(b), ref(r),
                                                                         ref(p)),
            lambda n: lib().bplx_simulate_tournament_paired(ref(s), ref(f), fake(50), fake(51), ref(t), ref(b), None,
                                                            ref(r), ref(p), *_draw_args(o), *_tournament_outputs(),
                                                            fake(60), None, None, None, None, None, None, fake(54),
                                                            None, n, None))


def _ppc_output(o):
    ptrs = {k: fake(70 + i) for i, k in enumerate(("score_counts", "outcome_counts", "goals", "total_goals_sq",
                                                   "team_points", "team_goals_for", "team_goals_against", "invalid"))}
    return _struct(_abi.PpcOutput, o, "out", scores=None, **ptrs)


def _ppc_args(o):
    return (o.get("max_goals", 10), o.get("score_bins", 6), o.get("pw", 3), o.get("pd", 1), o.get("R", 2),
            C.c_ulonglong(7), o.get("first_draw", 5))


def ppc(o, keep):
    s, obs, out = _samples(o), _observations(o), _ppc_output(o)
    return (lambda: lib().bplx_posterior_predictive_workspace_bytes(ref(s), ref(obs)),
            lambda n: lib().bplx_posterior_predictive(ref(s), ref(obs), *_ppc_args(o), ref(out), None, n, None))


def ppc_gameweeks(o, keep):
    s, obs, out, gw, ngw = _samples(o), _observations(o), _ppc_output(o), _gameweeks(o, keep), o.get("ngw", NGW)
    return (lambda: lib().bplx_posterior_predictive_gameweeks_workspace_bytes(ref(s), ngw, ref(obs)),
            lambda n: lib().bplx_posterior_predictive_gameweeks(ref(s), ngw, ref(obs), gw, *_ppc_args(o), ref(out),
                                                                None, n, None))


def lib():
    return _abi.lib()


CONSUMERS = {f.__name__: f for f in (score_grid, pointwise, pointwise_gameweeks, markets, table, table_conditional,
                                     tournament_ranked, tournament_paired, ppc, ppc_gameweeks)}

# workspace bytes of the valid shapes above
SIZES = {'markets': 670400,
 'pointwise': 543936,
 'pointwise_gameweeks': 532048,
 'ppc': 528128,
 'ppc_gameweeks': 528280,
 'score_grid': 767224,
 'table': 528128,
 'table_conditional': 533504,
 'tournament_paired': 531968,
 'tournament_ranked': 531968}


@pytest.mark.parametrize("name", sorted(CONSUMERS))
def test_size_call_matches_what_the_entry_point_needs(name):
    keep = []
    size, run = CONSUMERS[name]({}, keep)
    need = int(size())
    assert need == SIZES[name]
    assert run(need - 1) == _abi.E_WORKSPACE
    msg = lib().bplx_last_error().decode()
    assert msg == f"workspace too small: {need - 1} bytes given, {need} needed"


BIG = 2**62
# (consumer, overrides): the entry point's status and message, and the size call's bytes, for one fault each
MUTATIONS = {
    # max_goals in [1, 63]
    "grid_goals_0": ("score_grid", {"max_goals": 0}),
    "grid_goals_64": ("score_grid", {"max_goals": 64}),
    "markets_goals_0": ("markets", {"max_goals": 0}),
    "markets_goals_64": ("markets", {"max_goals": 64}),
    "table_goals_64": ("table", {"max_goals": 64}),
    "cup_goals_0": ("tournament_ranked", {"max_goals": 0}),
    "ppc_goals_64": ("ppc", {"max_goals": 64}),
    "ppc_gw_goals_0": ("ppc_gameweeks", {"max_goals": 0}),
    # points: 0 <= points_draw <= points_win, points_win >= 1
    "table_pw_0": ("table", {"t.points_win": 0, "t.points_draw": 0}),
    "table_pd_above_pw": ("table", {"t.points_draw": 4}),
    "cond_pd_negative": ("table_conditional", {"t.points_draw": -1}),
    "ppc_pw_0": ("ppc", {"pw": 0, "pd": 0}),
    "ppc_pd_negative": ("ppc", {"pd": -1}),
    "ppc_gw_pd_above_pw": ("ppc_gameweeks", {"pd": 4}),
    # draw range: sims_per_draw >= 1, (first_draw + S) R fits 63 bits, S R < 2^31
    "table_R_0": ("table", {"R": 0}),
    "table_first_negative": ("table", {"first_draw": -1}),
    "table_first_overflow": ("table", {"first_draw": BIG, "R": 2}),
    "table_SR_2_31": ("table", {"R": 3_000_000}),
    "paired_R_0": ("tournament_paired", {"R": 0}),
    "cup_SR_2_31": ("tournament_ranked", {"R": 3_000_000}),
    "ppc_R_0": ("ppc", {"R": 0}),
    "ppc_first_overflow": ("ppc", {"first_draw": BIG}),
    "ppc_SR_2_31": ("ppc", {"R": 3_000_000}),
    "ppc_gw_first_negative": ("ppc_gameweeks", {"first_draw": -1}),
    "ppc_gw_first_overflow": ("ppc_gameweeks", {"first_draw": BIG}),
    "ppc_gw_SR_2_31": ("ppc_gameweeks", {"R": 9_000_000}),
    # observed scores non-NULL
    "pointwise_no_home_goals": ("pointwise", {"obs.home_goals": None}),
    "pointwise_gw_no_away_goals": ("pointwise_gameweeks", {"obs.away_goals": None}),
    "ppc_no_home_goals": ("ppc", {"obs.home_goals": None}),
    "ppc_gw_no_away_goals": ("ppc_gameweeks", {"obs.away_goals": None}),
    # the predictive-check outputs
    "ppc_no_out": ("ppc", {"out": None}),
    "ppc_no_team_points": ("ppc", {"out.team_points": None}),
    "ppc_gw_no_invalid": ("ppc_gameweeks", {"out.invalid": None}),
    "ppc_no_obs": ("ppc", {"obs": None}),
    # size-call preconditions
    "grid_no_samples": ("score_grid", {"s": None}),
    "grid_no_fixtures": ("score_grid", {"f": None}),
    "pointwise_no_obs": ("pointwise", {"obs": None}),
    "pointwise_S_0": ("pointwise", {"s.num_samples": 0}),
    "pointwise_gw_ngw_0": ("pointwise_gameweeks", {"ngw": 0}),
    "pointwise_gw_ngw_3": ("pointwise_gameweeks", {"ngw": 3}),
    "pointwise_gw_F_0": ("pointwise_gameweeks", {"f.num_fixtures": 0}),
    "markets_no_lines": ("markets", {"lines": None}),
    "markets_T_0": ("markets", {"s.num_teams": 0}),
    "table_no_table": ("table", {"t": None}),
    "table_F_0": ("table", {"f.num_fixtures": 0}),
    "cup_F_0": ("tournament_ranked", {"f.num_fixtures": 0}),
    "cup_no_bracket": ("tournament_ranked", {"b": None}),
    "cup_groups_17": ("tournament_ranked", {"b.num_groups": 17}),
    "cup_best_negative": ("tournament_ranked", {"b.best_count": -1}),
    "paired_too_many": ("tournament_paired", {"p.num_pairings": 17}),
    "ppc_S_0": ("ppc", {"s.num_samples": 0}),
    "ppc_gw_ngw_7": ("ppc_gameweeks", {"ngw": 7}),
    "ppc_gw_T_0": ("ppc_gameweeks", {"s.num_teams": 0}),
    # ranking
    "cond_rule_5": ("table_conditional", {"r.rule": 5}),
    "cond_goal_diff": ("table_conditional", {"r.rule": _abi.RANK_GOAL_DIFF}),
    "cond_no_ranking": ("table_conditional", {"r": None}),
    "cond_h2h_slots_0": ("table_conditional", {"t.num_slots": 0}),
    "cond_goal_diff_slots_65": ("table_conditional", {"r.rule": _abi.RANK_GOAL_DIFF, "t.num_slots": 65}),
    "cup_rule_5": ("tournament_ranked", {"r.rule": 5}),
    "cup_h2h_slots_65": ("tournament_ranked", {"t.num_slots": 65}),
    "paired_goal_diff": ("tournament_paired", {"r.rule": _abi.RANK_GOAL_DIFF}),
    # two faults: the first check in order reports
    "ppc_goals_and_points": ("ppc", {"max_goals": 0, "pw": 0}),
    "ppc_gw_gameweek_and_goals": ("ppc_gameweeks", {"gameweek": np.full(F, NGW), "obs.home_goals": None}),
    "table_points_and_goals": ("table", {"t.points_win": 0, "max_goals": 0}),
    "table_goals_and_R": ("table", {"max_goals": 0, "R": 0}),
}

# (status, message, size call) of each mutation
EXPECTED = {'cond_goal_diff': (-5, 'workspace too small: 0 bytes given, 528128 needed', 528128),
 'cond_goal_diff_slots_65': (-2,
                             "simulate: 65 table slots exceed the kernel's limit of 64 (BPLX_SIM_MAX_TEAMS)",
                             528128),
 'cond_h2h_slots_0': (-1, 'simulate: the table needs at least one slot', 0),
 'cond_no_ranking': (-5, 'workspace too small: 0 bytes given, 528128 needed', 528128),
 'cond_pd_negative': (-1,
                      'simulate: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got 3, -1)',
                      533504),
 'cond_rule_5': (-1, 'simulate: ranking rule 5 is not a BPLX_RANK_* value', 0),
 'cup_F_0': (-5, 'workspace too small: 0 bytes given, 531968 needed', 531968),
 'cup_SR_2_31': (-2,
                 'tournament: num_samples * sims_per_draw must be below 2^31 per call (got 3000000000): cut the draws '
                 'into ranges',
                 531968),
 'cup_best_negative': (-2, 'tournament: best_count must be in [0, 16] (got -1)', 0),
 'cup_goals_0': (-1, 'tournament: max_goals must be in [1, 63] (got 0)', 531968),
 'cup_groups_17': (-1, 'tournament: num_groups must be in [0, num_slots] (got 17)', 0),
 'cup_h2h_slots_65': (-2, "tournament: 65 table slots exceed the kernel's limit of 64 (BPLX_SIM_MAX_TEAMS)", 0),
 'cup_no_bracket': (-1, 'tournament: bracket is NULL', 0),
 'cup_rule_5': (-1, 'tournament: ranking rule 5 is not a BPLX_RANK_* value', 0),
 'grid_goals_0': (-1, 'score grid: max_goals must be in [1, 63] (got 0)', 0),
 'grid_goals_64': (-1, 'score grid: max_goals must be in [1, 63] (got 64)', 8876728),
 'grid_no_fixtures': (-1, 'samples / fixtures is NULL', 0),
 'grid_no_samples': (-1, 'samples / fixtures is NULL', 0),
 'markets_T_0': (-1, 'markets: num_samples, num_teams and num_fixtures must be positive', 0),
 'markets_goals_0': (-1, 'markets: max_goals must be in [1, 63] (got 0)', 0),
 'markets_goals_64': (-1, 'markets: max_goals must be in [1, 63] (got 64)', 0),
 'markets_no_lines': (-1, 'markets: lines is NULL', 0),
 'paired_R_0': (-1, 'tournament: sims_per_draw must be >= 1 (got 0)', 531968),
 'paired_goal_diff': (-5, 'workspace too small: 0 bytes given, 528384 needed', 528384),
 'paired_too_many': (-1, 'pairings: num_pairings must be in [0, 16] (got 17)', 0),
 'pointwise_S_0': (-1, 'pointwise log-likelihood: num_samples, num_teams and num_fixtures must be positive', 0),
 'pointwise_gw_F_0': (-1,
                      'pointwise log-likelihood over gameweeks: num_samples, num_teams and num_fixtures must be '
                      'positive',
                      0),
 'pointwise_gw_ngw_0': (-1,
                        'pointwise log-likelihood over gameweeks: num_gameweeks (0) must be >= 1 and divide '
                        'num_samples (1000): the samples are gameweek-major',
                        0),
 'pointwise_gw_ngw_3': (-1,
                        'pointwise log-likelihood over gameweeks: num_gameweeks (3) must be >= 1 and divide '
                        'num_samples (1000): the samples are gameweek-major',
                        0),
 'pointwise_gw_no_away_goals': (-1,
                                'pointwise log-likelihood over gameweeks: home_goals and away_goals must not be NULL',
                                532048),
 'pointwise_no_home_goals': (-1, 'pointwise log-likelihood: home_goals and away_goals must not be NULL', 543936),
 'pointwise_no_obs': (-1, 'observations is NULL', 0),
 'ppc_R_0': (-1, 'posterior predictive: sims_per_draw must be >= 1 (got 0)', 528128),
 'ppc_SR_2_31': (-2,
                 'posterior predictive: num_samples * sims_per_draw must be below 2^31 per call (got 3000000000): cut '
                 'the draws into ranges',
                 528128),
 'ppc_S_0': (-1, 'posterior predictive: num_samples, num_teams and num_fixtures must be positive', 0),
 'ppc_first_overflow': (-1,
                        'posterior predictive: first_draw must be >= 0 and (first_draw + num_samples) * sims_per_draw '
                        'must fit 63 bits',
                        528128),
 'ppc_goals_64': (-1, 'posterior predictive: max_goals must be in [1, 63] (got 64)', 528128),
 'ppc_goals_and_points': (-1, 'posterior predictive: max_goals must be in [1, 63] (got 0)', 528128),
 'ppc_gw_SR_2_31': (-2,
                    'posterior predictive over gameweeks: draws * sims_per_draw must be below 2^31 per call (got '
                    '2250000000): cut the draws into ranges',
                    528280),
 'ppc_gw_T_0': (-1, 'posterior predictive over gameweeks: num_samples, num_teams and num_fixtures must be positive', 0),
 'ppc_gw_first_negative': (-1,
                           'posterior predictive over gameweeks: first_draw must be >= 0 and (first_draw + S) * '
                           'sims_per_draw must fit 63 bits',
                           528280),
 'ppc_gw_first_overflow': (-1,
                           'posterior predictive over gameweeks: first_draw must be >= 0 and (first_draw + S) * '
                           'sims_per_draw must fit 63 bits',
                           528280),
 'ppc_gw_gameweek_and_goals': (-1,
                               'posterior predictive over gameweeks: match 0 has gameweek 4 outside [0, 4)',
                               528280),
 'ppc_gw_goals_0': (-1, 'posterior predictive over gameweeks: max_goals must be in [1, 63] (got 0)', 528280),
 'ppc_gw_ngw_7': (-1,
                  'posterior predictive over gameweeks: num_gameweeks (7) must be >= 1 and divide num_samples (1000): '
                  'the samples are gameweek-major',
                  0),
 'ppc_gw_no_away_goals': (-1,
                          'posterior predictive over gameweeks: home_goals and away_goals must not be NULL',
                          528280),
 'ppc_gw_no_invalid': (-1, 'posterior predictive over gameweeks: every output but scores must be given', 528280),
 'ppc_gw_pd_above_pw': (-1,
                        'posterior predictive over gameweeks: points must satisfy 0 <= points_draw <= points_win, '
                        'points_win >= 1 (got 3, 4)',
                        528280),
 'ppc_no_home_goals': (-1, 'posterior predictive: home_goals and away_goals must not be NULL', 528128),
 'ppc_no_obs': (-1, 'posterior predictive: observations / out is NULL', 0),
 'ppc_no_out': (-1, 'posterior predictive: observations / out is NULL', 528128),
 'ppc_no_team_points': (-1, 'posterior predictive: every output but scores must be given', 528128),
 'ppc_pd_negative': (-1,
                     'posterior predictive: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got '
                     '3, -1)',
                     528128),
 'ppc_pw_0': (-1,
              'posterior predictive: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got 0, 0)',
              528128),
 'table_F_0': (-1, 'simulate: num_samples, num_teams and num_fixtures must be positive', 0),
 'table_R_0': (-1, 'simulate: sims_per_draw must be >= 1 (got 0)', 528128),
 'table_SR_2_31': (-2,
                   'simulate: num_samples * sims_per_draw must be below 2^31 per call (got 3000000000): cut the draws '
                   'into ranges',
                   528128),
 'table_first_negative': (-1,
                          'simulate: first_draw must be >= 0 and (first_draw + num_samples) * sims_per_draw must fit '
                          '63 bits',
                          528128),
 'table_first_overflow': (-1,
                          'simulate: first_draw must be >= 0 and (first_draw + num_samples) * sims_per_draw must fit '
                          '63 bits',
                          528128),
 'table_goals_64': (-1, 'simulate: max_goals must be in [1, 63] (got 64)', 528128),
 'table_goals_and_R': (-1, 'simulate: max_goals must be in [1, 63] (got 0)', 528128),
 'table_no_table': (-1, 'simulate: table is NULL', 0),
 'table_pd_above_pw': (-1,
                       'simulate: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got 3, 4)',
                       528128),
 'table_points_and_goals': (-1,
                            'simulate: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got 0, 1)',
                            528128),
 'table_pw_0': (-1, 'simulate: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got 0, 0)', 528128)}


@pytest.mark.parametrize("case", sorted(MUTATIONS))
def test_one_fault_gives_the_recorded_status_text_and_size(case):
    name, o = MUTATIONS[case]
    keep = []
    size, run = CONSUMERS[name](o, keep)
    status = run(0)
    msg = lib().bplx_last_error().decode() if status != _abi.OK else ""
    want_status, want_msg, want_size = EXPECTED[case]
    assert status == want_status
    if case.startswith("grid_goals"):  # the score grid's message gained the "score grid: " prefix the others have
        assert msg in (want_msg, want_msg.removeprefix("score grid: "))
    else:
        assert msg == want_msg
    assert int(size()) == want_size
