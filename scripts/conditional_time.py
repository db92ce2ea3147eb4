"""Times match importance (bplx_simulate_table_conditional) on one GPU against the plain table call on the same inputs.

    python scripts/conditional_time.py [--samples 16384] [--sims-per-draw 64] [--reps 20] [--out FILE.json]

Workloads, each under both ranking rules:
  league_10x60   the F = 380 league of 20 teams, Kc = 10 key fixtures, E = 60 events (title, top four and relegation
                 for every team);
  league_64x64   the same league with Kc = E = 64;
  wc48_24x48     the 48-team group stage (12 groups of four, 72 fixtures, NeutralWC at neutral venues), Kc = 24 (the
                 last round) and E = 48 (each team in the top two of its group).
S draws x R simulations per draw (default 16,384 x 64 = 2^20 seasons).  Each call is timed with CUDA events over
--reps calls after a warm-up call, best of three rounds alternating the plain and the conditional call.  The plain call
runs the unchanged kernels.  Reports the GPU name, power limit and max SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from simulate_time import gpu_info  # noqa: E402


def league(S):
    from bpl_next_b200 import season
    from tests.test_score_grid_gpu import make_samples

    s = make_samples("dixon_coles", S, 20, 4, seed=7)
    names = [f"T{i:02d}" for i in range(20)]
    tab = season.build_table(names)
    pairs = [(i, j) for i in range(20) for j in range(20) if i != j]
    hs, as_ = season.fixture_slots(tab, [names[i] for i, _ in pairs], [names[j] for _, j in pairs])
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16)}
    return "dixon_coles", s, fx, hs, as_, tab, names


def wc48(S):
    from bpl_next_b200 import season
    from tests.test_score_grid_gpu import make_samples

    s = make_samples("neutral_wc", S, 48, 6, seed=61)
    names = [f"T{i:02d}" for i in range(48)]
    tab = season.build_table(names, groups=[chr(65 + i // 4) for i in range(48)])
    # rounds of a group of four: (0 1, 2 3), (0 2, 1 3), (0 3, 1 2); the last round is fixtures 48..71
    rounds = [((0, 1), (2, 3)), ((0, 2), (1, 3)), ((0, 3), (1, 2))]
    pairs = [(4 * g + a, 4 * g + b) for rnd in rounds for g in range(12) for a, b in rnd]
    hs, as_ = season.fixture_slots(tab, [names[i] for i, _ in pairs], [names[j] for _, j in pairs])
    fx = {"home_team": hs.astype(np.uint16), "away_team": as_.astype(np.uint16),
          "neutral_venue": np.ones(len(pairs), np.uint8), "home_conf": (hs % 6).astype(np.uint8),
          "away_conf": (as_ % 6).astype(np.uint8)}
    return "neutral_wc", s, fx, hs, as_, tab, names


def workloads(S):
    lg, wc = league(S), wc48(S)
    names = lg[-1]
    ev60 = {}
    for t in names:
        ev60.update({f"{t} title": (t, 0), f"{t} top4": (t, range(4)), f"{t} down": (t, (17, 18, 19))})
    ev64 = dict(ev60, **{f"{t} europe": (t, range(4, 6)) for t in names[:4]})
    return [("league_10x60", lg, list(range(370, 380)), ev60), ("league_64x64", lg, list(range(316, 380)), ev64),
            ("wc48_24x48", wc, list(range(48, 72)), {f"{t} through": (t, (0, 1)) for t in wc[-1]})]


def main():
    import torch

    from bpl_next_b200 import problem, season

    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--sims-per-draw", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    a = ap.parse_args()
    S, R = a.samples, a.sims_per_draw
    res = {"gpu": gpu_info(), "samples": S, "sims_per_draw": R, "simulations": S * R}
    dev = lambda d: {k: None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in d.items()}
    for name, (model, s, fx, hs, as_, tab, _), keys, events in workloads(S):
        c = season.build_conditions(tab, len(hs), keys, events)
        (g,) = c["groups"]
        cond = dict(g, event_slot=c["event_slot"], event_positions=c["event_positions"])
        ds, dfx = dev(s), dev(dict(fx, home_slot=hs, away_slot=as_))
        for rule in ("goal_difference", "head_to_head"):
            dtab = dev({k: tab[k] for k in ("start_points", "start_goals_for", "start_goals_against", "group")})
            dtab.update({k: tab[k] for k in ("num_positions", "num_points_bins", "points_win", "points_draw")},
                        tiebreak=rule, played_h2h=None)
            ws = torch.empty(1 << 28, dtype=torch.uint8, device="cuda")
            calls = {"plain": lambda: problem.simulate_table(model, ds, dfx, dtab, 15, R, 7, workspace=ws),
                     "conditional": lambda: problem.simulate_table(model, ds, dfx, dtab, 15, R, 7, workspace=ws,
                                                                   conditions=cond)}
            best = {k: float("inf") for k in calls}
            for _ in range(3):
                for k, call in calls.items():
                    out = call()
                    assert int(out["invalid"].item()) == 0, (name, rule, k)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(a.reps):
                        call()
                    e1.record()
                    torch.cuda.synchronize()
                    best[k] = min(best[k], e0.elapsed_time(e1) / a.reps)
            p, q = calls["plain"](), calls["conditional"]()
            for k in ("position_counts", "points_counts"):
                assert torch.equal(p[k], q[k]), (name, rule, k)
            row = {"key_fixtures": len(keys), "events": len(events), "plain_ms": round(best["plain"], 4),
                   "conditional_ms": round(best["conditional"], 4),
                   "added": round(best["conditional"] / best["plain"] - 1.0, 4)}
            res[f"{name}_{rule}"] = row
            print(name, rule, row, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
