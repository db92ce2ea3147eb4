"""Times tournament simulation (bplx_simulate_tournament) on one GPU against the group stage alone.

    python scripts/tournament_time.py [--samples 16384] [--reps 20] [--out FILE.json]

Workloads (synthetic posterior draws, fixed seeds):
  world cup  the 48-team format: simulate_time.py's 12 groups of four (72 neutral fixtures, NeutralWC draws of
             configs[5]'s shape), the 8 best thirds through a generated complete 495-row allocation table, a round of
             32, 16, QF, SF, a third-place match and the final (32 neutral ties); R = 64 and R = 1.  The same call of
             bplx_simulate_table (group stage only) is timed in the same run, so the cost per (simulation, tie) is
             (tournament - group stage) / (N K).
  knockout   16 teams, no group stage (F = 0), 15 ties + a third-place match, NeutralWC draws of configs[5]'s
             shape, R = 64.
CUDA events around `--reps` calls after warm-up; a call is the whole entry point (count resets, exponential-table
pre-pass, kernel), issued straight through the C ABI.  Reports the GPU name and power limit read in the same run and
the shared memory per CTA of both kernels at the world-cup shape.
"""
from __future__ import annotations

import argparse
import ctypes as C
import itertools
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.dont_write_bytecode = True

from simulate_time import device_table, gpu_info, prepared_call, time_ms, world_cup  # noqa: E402


def _knockout(entrants):
    """Pairs in order, then the winners round by round; a third-place match before the final."""
    ties, prev, r = [], list(entrants), 0
    while len(prev) > 1:
        cur = []
        for k in range(0, len(prev), 2):
            ties.append({"id": f"t{len(ties)}", "round": f"r{r}", "home": prev[k], "away": prev[k + 1],
                         "neutral_venue": 1})
            cur.append(("winner", ties[-1]["id"]))
        if len(cur) == 1:
            final = ties.pop()
            ties.append({"id": "third", "round": "third", "home": ("loser", final["home"][1]),
                         "away": ("loser", final["away"][1]), "neutral_venue": 1})
            ties.append(final)
        prev, r = cur, r + 1
    return ties


def world_cup_bracket(teams, group):
    from bpl_next_b200 import season

    names = [f"S{i}" for i in range(48)]
    L = [f"g{g:02d}" for g in range(12)]
    tab = season.build_table(names, groups=[L[g] for g in group])
    alloc = {}
    for sub in itertools.combinations(L, 8):
        r = len(alloc) % 8
        alloc[frozenset(sub)] = list(sub[r:] + sub[:r])
    ent = [("group", g, 0) for g in L] + [("group", g, 1) for g in L] + [("best", j) for j in range(8)]
    br = season.build_bracket(tab, _knockout(ent), {"position": 2, "count": 8, "allocation": alloc})
    br["slot_team"] = teams.astype(np.uint16)
    br["slot_conf"] = (teams % 6).astype(np.uint8)
    return br


def tournament_call(model, s, fx, hs, as_, T_tab, group, br, R, seed=1):
    """The bplx_simulate_tournament call with every argument built once; returns (call, outputs, keep-alive)."""
    import torch

    from bpl_next_b200 import _abi, problem

    lib = _abi.lib()
    keep = []
    ptr = problem._device_ptr_fn(keep)
    dev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    st = problem._samples_struct(model, dev, ptr)
    F = len(hs)
    if F:
        dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fx.items()}
        ft = problem._fixtures_struct(dfx, ptr)
        d_hs, d_as = ptr(torch.from_numpy(hs).cuda()), ptr(torch.from_numpy(as_).cuda())
    else:
        ft, d_hs, d_as = _abi.Fixtures(), None, None
    tab = device_table(T_tab, group, hs, as_)
    t = problem._table_struct(tab, ptr)
    b = problem._bracket_struct(br, keep)
    cnt = {k: torch.empty(n, dtype=torch.int64, device="cuda") for k, n in
           (("pos", T_tab * t.num_positions), ("pts", T_tab * t.num_points_bins), ("reach", T_tab * b.num_rounds),
            ("win", T_tab * b.num_rounds), ("invalid", 1))}
    need = int(lib.bplx_simulate_tournament_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t), C.byref(b)))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    args = (C.byref(st), C.byref(ft), d_hs, d_as, C.byref(t), C.byref(b), 15, R, seed, 0, ptr(cnt["pos"]),
            ptr(cnt["pts"]), ptr(cnt["reach"]), ptr(cnt["win"]), None, None, None, None, None, ptr(cnt["invalid"]),
            ptr(ws), ws.numel(), stream)

    def call():
        _abi.check(lib.bplx_simulate_tournament(*args))

    return call, cnt, (keep, st, ft, t, b, dev, tab, ws)


def smem_bytes(T_tab, P, B, nr=0, K=0):
    """simulate_smem_bytes (csrc/simulate.cu) for a table of T_tab slots; nr, K > 0: the tournament kernel."""
    base = T_tab * 128 * 16 + T_tab * P * 4 + T_tab * 12 + T_tab * B * 4
    if K:
        base += T_tab * nr * 8 + (0 if K <= 4 * T_tab else (2 * K + 3) // 4 * 4 * 128)
    return base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from oracle import datasets

    if not torch.cuda.is_available():
        raise SystemExit("tournament_time.py measures the GPU kernel and needs a CUDA device")
    S = a.samples
    rows = []
    model, s, fx, hs, as_, T_tab, group = world_cup(S)
    rng = np.random.default_rng(11)
    teams = rng.choice(220, 48, replace=False)  # world_cup()'s slot -> team map (same seed, same draw)
    assert np.array_equal(teams[hs], fx["home_team"])
    br = world_cup_bracket(teams, group)
    K = len(br["round"])
    for R in (64, 1):
        gcall, gout, _gk = prepared_call(model, s, fx, hs, as_, T_tab, group, R)
        tcall, tout, _tk = tournament_call(model, s, fx, hs, as_, T_tab, group, br, R)
        for _ in range(3):
            gcall()
            tcall()
        torch.cuda.synchronize()
        assert int(gout["invalid"].item()) == 0 and int(tout["invalid"].item()) == 0
        assert torch.equal(gout["position_counts"].flatten(), tout["pos"])
        ms_g, ms_t = [], []
        for _ in range(3):  # alternate the two calls
            ms_g.append(time_ms(gcall, a.reps))
            ms_t.append(time_ms(tcall, a.reps))
        g, t = min(ms_g), min(ms_t)
        N, F = S * R, len(hs)
        rows.append({"workload": "world cup 48, 12 groups + 32 ties", "model": model, "S": S, "R": R, "N": N, "F": F,
                     "K": K, "group_stage_ms": g, "tournament_ms": t, "group_stage_ms_all": ms_g,
                     "tournament_ms_all": ms_t, "ps_per_sim_fixture": g * 1e9 / (N * F),
                     "ps_per_sim_tie": (t - g) * 1e9 / (N * K), "tournaments_per_s": N / (t * 1e-3)})
        print(json.dumps(rows[-1]), flush=True)
    # 16 teams, no group stage
    s16, _ = datasets.config_5(S=S, F=1)
    s16 = {k: v for k, v in s16.items()}
    from bpl_next_b200 import season

    names = [f"S{i}" for i in range(16)]
    tab = season.build_table(names)
    br16 = season.build_bracket(tab, _knockout([("team", n) for n in names]))
    br16["slot_team"] = np.arange(0, 160, 10).astype(np.uint16)
    br16["slot_conf"] = (br16["slot_team"] % 6).astype(np.uint8)
    e = np.zeros(0, np.uint8)
    for R in (64,):
        call, out, _k = tournament_call("neutral_wc", s16, {}, e, e, 16, None, br16, R)
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        assert int(out["invalid"].item()) == 0
        ms = min(time_ms(call, a.reps) for _ in range(3))
        N, K16 = S * R, len(br16["round"])
        rows.append({"workload": "knockout only, 16 teams, 16 ties", "model": "neutral_wc", "S": S, "R": R, "N": N,
                     "F": 0, "K": K16, "tournament_ms": ms, "ps_per_sim_tie": ms * 1e9 / (N * K16),
                     "tournaments_per_s": N / (ms * 1e-3)})
        print(json.dumps(rows[-1]), flush=True)
    P, B = 4, 3 * 3 + 1
    res = {"gpu": gpu_info(), "reps": a.reps, "workloads": rows,
           "smem_bytes_world_cup": {"group_stage": smem_bytes(48, P, B),
                                    "tournament": smem_bytes(48, P, B, br["num_rounds"], K),
                                    "histograms": 48 * br["num_rounds"] * 8}}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
