"""Times tournaments with pairings drawn by lot (bplx_simulate_tournament_paired) on one GPU against the same
brackets with their pairs fixed.

    python scripts/pairing_time.py [--samples 16384] [--sims-per-draw 64] [--reps 20] [--out FILE.json]

Workloads (NeutralWC draws of configs[5]'s shape, fixed seeds):
  cup   64 teams, no group stage (F = 0), an open draw before every round: 6 pairings (64, 32, .. 2 entrants) and 63
        one-match ties.
  uefa  32 teams in 8 groups of four ranked head-to-head (96 fixtures, each pair of a group home and away), a seeded
        round of 16 of the group winners against the runners-up under group and association protection, open
        quarter- and semi-final draws, all two-legged, and a one-match final with extra time at a neutral venue: 3
        pairings and 15 ties.
Each workload is timed alternating with the same bracket whose ties take fixed entrants (pool order: pair i = entrants
2i and 2i + 1 of an open pool, runner-up i against winner i of a seeded one), so (paired - fixed) / (N P) is the cost
of one pairing per simulation.  A call is problem.simulate_tournament on device tensors (count resets, the
exponential-table pre-pass, the kernel, and the host's argument checks); CUDA events around `--reps` calls after
warm-up, best of three alternating rounds.  Reports the GPU name and power limit read in the same run.
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
sys.dont_write_bytecode = True

from simulate_time import gpu_info  # noqa: E402


def _rounds(first, n, fixed):
    """Ties of a knockout whose every round after the first is an open draw (or, fixed, the winners in order)."""
    ties, pairings, prev, r = [], [], None, 0
    while n > 1:
        ids = [f"r{r}_{i}" for i in range(n // 2)]
        if prev is None:
            pool = first
        else:
            pool = [("winner", t) for t in prev]
        if fixed:
            ties += [{"id": t, "round": f"r{r}", "home": pool[2 * i], "away": pool[2 * i + 1]} for i, t in enumerate(ids)]
        else:
            pairings.append({"id": f"d{r}", "pool": pool, "pots": None})
            ties += [{"id": t, "round": f"r{r}", "pair": (f"d{r}", i)} for i, t in enumerate(ids)]
        prev, n, r = ids, n // 2, r + 1
    return ties, pairings


def cup(fixed):
    names = [f"S{i}" for i in range(64)]
    ties, pairings = _rounds([("team", t) for t in names], 64, fixed)
    return names, None, {}, ties, pairings, None


def uefa(fixed):
    names = [f"S{i}" for i in range(32)]
    L = "ABCDEFGH"
    groups = [L[i // 4] for i in range(32)]
    hs = [4 * g + i for g in range(8) for i in range(4) for j in range(4) if i != j]
    as_ = [4 * g + j for g in range(8) for i in range(4) for j in range(4) if i != j]
    fx = {"home": [names[i] for i in hs], "away": [names[i] for i in as_]}
    assoc = [f"N{i // 8}" for i in range(32)]
    W, R = [("group", g, 0) for g in L], [("group", g, 1) for g in L]
    if fixed:
        ties = [{"id": f"r16_{i}", "round": "R16", "home": R[i], "away": W[i], "format": "two_legs"} for i in range(8)]
        pairings = []
    else:
        ties = [{"id": f"r16_{i}", "round": "R16", "pair": ("r16", i), "format": "two_legs"} for i in range(8)]
        pairings = [{"id": "r16", "pool": W + R, "pots": [0] * 8 + [1] * 8, "protect": {"group", "association"}}]
    later, more = _rounds([("winner", f"r16_{i}") for i in range(8)], 8, fixed)
    for t in later:
        t["format"] = "two_legs"
        t["round"] = "x" + t["round"]
        if "pair" in t:
            t["pair"] = ("x" + t["pair"][0], t["pair"][1])
    for p in more:
        p["id"] = "x" + p["id"]
    later[-1] = {"id": later[-1]["id"], "round": "F", "home": ("winner", later[-3]["id"]),
                 "away": ("winner", later[-2]["id"]), "format": "extra_time", "neutral_venue": 1}
    return names, groups, fx, ties + later, pairings + more[:2], assoc


def build(workload, fixed, S, R):
    import torch

    from bpl_next_b200 import season
    from oracle import datasets

    names, groups, fx, ties, pairings, assoc = workload(fixed)
    s, _ = datasets.config_5(S=S, F=1)
    teams = np.random.default_rng(17).choice(220, len(names), replace=False)
    conf = (teams % 6).astype(np.uint8)
    tab = season.build_table(names, groups=groups, tiebreak="head_to_head" if groups else "goal_difference")
    dfx = {}
    if fx:
        hs, as_ = season.fixture_slots(tab, fx["home"], fx["away"])
        arr = {"home_team": teams[hs].astype(np.uint16), "away_team": teams[as_].astype(np.uint16),
               "home_conf": conf[hs], "away_conf": conf[as_], "neutral_venue": np.zeros(len(hs), np.uint8),
               "home_slot": hs, "away_slot": as_}
        dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in arr.items()}
    else:
        season._size_histograms(tab)
    br = season.build_bracket(tab, ties, pairings=pairings or None, association=assoc)
    br["slot_team"] = teams.astype(np.uint16)
    br["slot_conf"] = conf
    ds = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    dtab = {k: None if tab[k] is None else torch.from_numpy(tab[k]).cuda()
            for k in ("start_points", "start_goals_for", "start_goals_against", "group")}
    dtab.update({k: tab[k] for k in ("num_positions", "num_points_bins", "points_win", "points_draw", "tiebreak")})
    dtab["played_h2h"] = tab.get("played_h2h")
    ws = torch.empty(1 << 28, dtype=torch.uint8, device="cuda")
    return ds, dfx, dtab, br, ws, len(pairings)


def main():
    import torch

    from bpl_next_b200 import problem

    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--sims-per-draw", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    a = ap.parse_args()
    S, R = a.samples, a.sims_per_draw
    N = S * R
    res = {"gpu": gpu_info(), "samples": S, "sims_per_draw": R, "simulations": N}
    for name, wl in (("cup", cup), ("uefa", uefa)):
        calls = {}
        for fixed in (False, True):
            ds, dfx, dtab, br, ws, P = build(wl, fixed, S, R)
            calls[fixed] = (lambda ds=ds, dfx=dfx, dtab=dtab, br=br, ws=ws: problem.simulate_tournament(
                "neutral_wc", ds, dfx, dtab, br, 15, R, 7, workspace=ws), P)
        best = {False: float("inf"), True: float("inf")}
        for _ in range(3):
            for fixed in (False, True):
                call = calls[fixed][0]
                out = call()
                assert int(out["invalid"].item()) == 0, (name, fixed)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    call()
                e1.record()
                torch.cuda.synchronize()
                best[fixed] = min(best[fixed], e0.elapsed_time(e1) / a.reps)
        P = calls[False][1]
        res[name] = {"pairings": P, "paired_ms": round(best[False], 4), "fixed_ms": round(best[True], 4),
                     "per_pairing_ns": round((best[False] - best[True]) * 1e6 / (N * P), 4)}
        print(name, res[name], flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
