"""Restatement of match importance in season / group-stage simulation (``csrc/simulate_cond.cu``) in integer numpy.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  It builds on ``oracle/simulate.py`` and
``oracle/head_to_head.py`` (the same Philox words, score walks and rankings) and counts their positions, scores and
validity.

Definition (the same text as ``include/bplx.h``):

* Key fixtures: 1 <= Kc <= 64 distinct indices into the call's F fixtures.  In a simulation, key fixture j has outcome
  o in {0 home win, 1 draw, 2 away win}, taken from its sampled score (hg > ag, hg = ag, hg < ag).
* Events: 1 <= E <= 64.  Event e is a pair (slot t_e, position set M_e); M_e is a uint64 bit mask over 0-based positions
  within t_e's group.  Event e holds in a simulation iff t_e's position is in M_e.
* ``outcome_counts [Kc, 3]``: valid simulations in which key fixture j ended in outcome o.
  ``conditional_counts [Kc, 3, E]``: valid simulations in which key fixture j ended in o and event e held.  Invalid
  simulations are excluded exactly as they are from ``position_counts``.
* No random word is added or moved: every other output is the simulation's without conditions.
"""
from __future__ import annotations

import numpy as np

from oracle import head_to_head as h2h
from oracle import simulate as osim


def outcomes(home, away):
    """Outcome codes ``[n, F]``: 0 home win, 1 draw, 2 away win."""
    home, away = np.asarray(home, np.int64), np.asarray(away, np.int64)
    return np.where(home > away, 0, np.where(home == away, 1, 2))


def events(positions, event_slot, event_positions):
    """``[n, E]`` bool: event e holds (slot ``event_slot[e]``'s position is a bit of ``event_positions[e]``)."""
    pos = np.asarray(positions, np.int64)[:, np.asarray(event_slot, np.int64)]  # [n, E]
    masks = np.asarray(event_positions, np.uint64)[None, :]
    return ((masks >> np.minimum(pos, 63).astype(np.uint64)) & np.uint64(1)).astype(bool) & (pos < 64)


def counts(home, away, positions, valid, key_fixture, event_slot, event_positions):
    """``outcome_counts [Kc, 3]`` and ``conditional_counts [Kc, 3, E]`` (int64) of simulations with scores ``home`` /
    ``away [n, F]``, positions ``[n, T]`` and validity ``valid [n]``."""
    valid = np.asarray(valid, bool)
    keys = np.asarray(key_fixture, np.int64)
    out = outcomes(np.asarray(home)[:, keys][valid], np.asarray(away)[:, keys][valid])  # [v, Kc]
    ev = events(np.asarray(positions)[valid], event_slot, event_positions)  # [v, E]
    onehot = (out[:, :, None] == np.arange(3)[None, None, :]).reshape(len(out), -1)  # [v, Kc 3]
    # (a float64 product is exact: every count is below 2^53)
    cond = np.rint(onehot.T.astype(np.float64) @ ev.astype(np.float64)).astype(np.int64)
    Kc = len(keys)
    return onehot.sum(axis=0).reshape(Kc, 3).astype(np.int64), cond.reshape(Kc, 3, -1)


def simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed, conditions,
             first_draw=0, tiebreak="goal_difference", played_h2h=None):
    """The simulations of ``oracle.simulate.simulate`` (``oracle.head_to_head.simulate`` under ``"head_to_head"``)
    with ``conditions`` (``key_fixture``, ``event_slot``, ``event_positions``): its outputs plus ``outcome_counts`` and
    ``conditional_counts``."""
    if tiebreak == "goal_difference":
        out = osim.simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed,
                            first_draw)
    else:
        out = h2h.simulate(model, samples, fixtures, home_slot, away_slot, table, max_goals, sims_per_draw, seed,
                           first_draw, tiebreak, played_h2h)
    oc, cc = counts(out["home"], out["away"], out["positions"], out["valid"], conditions["key_fixture"],
                    conditions["event_slot"], conditions["event_positions"])
    out.update(outcome_counts=oc, conditional_counts=cc)
    return out
