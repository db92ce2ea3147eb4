"""Times tournament simulation (bplx_simulate_tournament) on one GPU against the group stage alone.

    python scripts/tournament_time.py [--samples 16384] [--reps 20] [--baseline-lib OLD/libbplx.so] [--out FILE.json]

Workloads (synthetic posterior draws, fixed seeds):
  world cup  the 48-team format: simulate_time.py's 12 groups of four (72 neutral fixtures, NeutralWC draws of
             configs[5]'s shape), the 8 best thirds through a generated complete 495-row allocation table, a round of
             32, 16, QF, SF, a third-place match and the final (32 neutral ties); R = 64 and R = 1.  The same call of
             bplx_simulate_table (group stage only) is timed in the same run, so the cost per (simulation, tie) is
             (tournament - group stage) / (N K).
  knockout   16 teams, no group stage (F = 0), 15 ties + a third-place match, NeutralWC draws of configs[5]'s
             shape, R = 64.
  champions league  the 2024 format: a 36-team league phase (144 fixtures, every team 4 at home and 4 away, NeutralWC
             draws of configs[5]'s shape, no neutral venues), a play-off round 24 v 9 .. 17 v 16, a round of 16 of its
             winners against the top 8, QF and SF, all two-legged (8 + 8 + 4 + 2 ties, the lower-placed or unseeded team
             at home first), and a one-match final with extra time at a neutral venue; R = 64.  The same bracket with
             every tie a single match (format 0) and the league phase alone run in the same run, so a two-legged tie is
             priced against a one-match tie per (simulation, tie).
The world-cup calls go through bplx_simulate_tournament_ex (tie_format all 0, decided_counts on: what
problem.simulate_tournament issues).  With --baseline-lib, another build's bplx_simulate_tournament is timed on the
same world-cup call, alternating with this build's, and its counts are checked equal.  The world-cup group stage and
tournament are also timed under the head-to-head ranking rule (bplx_simulate_table_ex / _tournament_ranked, no played
matches), alternating with the goal-difference calls in the same run: h2h_*_ms and h2h_*_cost.
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

from simulate_time import baseline_lib, device_table, gpu_info, prepared_call, time_ms, world_cup  # noqa: E402


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


def champions_league_ties():
    """The 2024 Champions League knockout on a 36-position league table: play-off round (24 v 9 .. 17 v 16), round of
    16 (play-off winners v the top 8), QF, SF, all two-legged with the lower-placed or unseeded team at home first, and
    a one-match final with extra time at a neutral venue: 23 ties."""
    pos = lambda p: ("group", None, p)  # noqa: E731
    ties = [{"id": f"po{i}", "round": "PO", "home": pos(23 - i), "away": pos(8 + i), "format": "two_legs"}
            for i in range(8)]
    ties += [{"id": f"r{i}", "round": "R16", "home": ("winner", f"po{i}"), "away": pos(7 - i), "format": "two_legs"}
             for i in range(8)]
    ties += [{"id": f"q{i}", "round": "QF", "home": ("winner", f"r{2 * i}"), "away": ("winner", f"r{2 * i + 1}"),
              "format": "two_legs"} for i in range(4)]
    ties += [{"id": f"s{i}", "round": "SF", "home": ("winner", f"q{2 * i}"), "away": ("winner", f"q{2 * i + 1}"),
              "format": "two_legs"} for i in range(2)]
    ties.append({"id": "f", "round": "F", "home": ("winner", "s0"), "away": ("winner", "s1"), "neutral_venue": 1,
                 "format": "extra_time"})
    return ties


def champions_league(S):
    """36 of configs[5]'s teams; league phase: slot t hosts t + 1 .. t + 4 (mod 36), 144 fixtures, no neutral venue."""
    from bpl_next_b200 import season
    from oracle import datasets

    s, _ = datasets.config_5(S=S, F=1)
    teams = np.random.default_rng(13).choice(220, 36, replace=False)
    hs = np.repeat(np.arange(36), 4)
    as_ = (hs + np.tile(np.arange(1, 5), 36)) % 36
    conf = (teams % 6).astype(np.uint8)
    fx = {"home_team": teams[hs].astype(np.uint16), "away_team": teams[as_].astype(np.uint16),
          "home_conf": conf[hs], "away_conf": conf[as_], "neutral_venue": np.zeros(len(hs), np.uint8)}
    br = season.build_bracket(season.build_table([f"S{i}" for i in range(36)]), champions_league_ties())
    br["slot_team"] = teams.astype(np.uint16)
    br["slot_conf"] = conf
    return s, fx, hs.astype(np.uint8), as_.astype(np.uint8), br


def tournament_call(model, s, fx, hs, as_, T_tab, group, br, R, seed=1, lib=None, head_to_head=False):
    """The bplx_simulate_tournament_ex call (the bracket's tie_format, decided_counts on) with every argument built once;
    returns (call, outputs, keep-alive).  ``lib``: another build's library, called through its bplx_simulate_tournament.
    ``head_to_head``: bplx_simulate_tournament_ranked under that ranking rule."""
    import torch

    from bpl_next_b200 import _abi, problem

    legacy = lib is not None
    lib = _abi.lib() if lib is None else lib
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
            ("win", T_tab * b.num_rounds), ("decided", 3 * b.num_ties), ("invalid", 1))}
    rk = _abi.Ranking(_abi.RANK_HEAD_TO_HEAD, None)
    if head_to_head:
        need = int(lib.bplx_simulate_tournament_ranked_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t),
                                                                        C.byref(b), C.byref(rk)))
    else:
        need = int(lib.bplx_simulate_tournament_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t), C.byref(b)))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    head = (C.byref(st), C.byref(ft), d_hs, d_as, C.byref(t), C.byref(b))
    tail = (ptr(cnt["invalid"]), ptr(ws), ws.numel(), stream)
    if legacy:
        fn, args = lib.bplx_simulate_tournament, head + (15, R, seed, 0, ptr(cnt["pos"]), ptr(cnt["pts"]),
                                                         ptr(cnt["reach"]), ptr(cnt["win"]), None, None, None, None,
                                                         None) + tail
    else:
        fmt = np.ascontiguousarray(br["tie_format"], np.uint8)
        keep.append(fmt)
        fn, args = lib.bplx_simulate_tournament_ex, head + (fmt.ctypes.data, 15, R, seed, 0, ptr(cnt["pos"]),
                                                            ptr(cnt["pts"]), ptr(cnt["reach"]), ptr(cnt["win"]),
                                                            ptr(cnt["decided"]), None, None, None, None, None,
                                                            None) + tail
        if head_to_head:
            fn, args = lib.bplx_simulate_tournament_ranked, args[:7] + (C.byref(rk),) + args[7:]

    def call():
        rc = fn(*args)
        if rc != _abi.OK:
            raise _abi.BplxError(rc, lib.bplx_last_error().decode("utf-8", "replace"))

    return call, cnt, (keep, st, ft, t, b, dev, tab, ws, rk)


def smem_bytes(T_tab, P, B, nr=0, K=0):
    """simulate_smem_bytes (csrc/simulate.cu) for a table of T_tab slots; nr, K > 0: the tournament kernel."""
    base = T_tab * 128 * 16 + T_tab * P * 4 + T_tab * 12 + T_tab * B * 4
    if K:
        base += T_tab * nr * 8 + K * 8 + (0 if K <= 4 * T_tab else (2 * K + 3) // 4 * 4 * 128)
    return base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--baseline-lib", default=None, help="another build's libbplx.so, timed on the world-cup call")
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
    base = None
    if a.baseline_lib:
        base = baseline_lib(a.baseline_lib, ("bplx_simulate_tournament", "bplx_simulate_tournament_workspace_bytes",
                                             "bplx_last_error"))
    for R in (64, 1):
        gcall, gout, _gk = prepared_call(model, s, fx, hs, as_, T_tab, group, R)
        tcall, tout, _tk = tournament_call(model, s, fx, hs, as_, T_tab, group, br, R)
        calls = [gcall, tcall]
        if base is not None:
            bcall, bout, _bk = tournament_call(model, s, fx, hs, as_, T_tab, group, br, R, lib=base)
            calls.append(bcall)
        # the group stage and the tournament under the head-to-head rule: the last two calls
        hgcall, hgout, _hgk = prepared_call(model, s, fx, hs, as_, T_tab, group, R, head_to_head=True)
        htcall, htout, _htk = tournament_call(model, s, fx, hs, as_, T_tab, group, br, R, head_to_head=True)
        calls += [hgcall, htcall]
        for _ in range(3):
            for c in calls:
                c()
        torch.cuda.synchronize()
        assert int(gout["invalid"].item()) == 0 and int(tout["invalid"].item()) == 0
        assert int(hgout["invalid"].item()) == 0 and int(htout["invalid"].item()) == 0
        assert torch.equal(hgout["position_counts"].flatten(), htout["pos"])
        assert torch.equal(gout["position_counts"].flatten(), tout["pos"])
        if base is not None:
            for k in ("pos", "pts", "reach", "win", "invalid"):
                assert torch.equal(tout[k], bout[k]), k
        ms = [[] for _ in calls]
        for _ in range(3):  # alternate the calls
            for c, m in zip(calls, ms):
                m.append(time_ms(c, a.reps))
        g, t = min(ms[0]), min(ms[1])
        N, F = S * R, len(hs)
        rows.append({"workload": "world cup 48, 12 groups + 32 ties", "model": model, "S": S, "R": R, "N": N, "F": F,
                     "K": K, "group_stage_ms": g, "tournament_ms": t, "group_stage_ms_all": ms[0],
                     "tournament_ms_all": ms[1], "ps_per_sim_fixture": g * 1e9 / (N * F),
                     "ps_per_sim_tie": (t - g) * 1e9 / (N * K), "tournaments_per_s": N / (t * 1e-3)})
        if base is not None:
            rows[-1].update(baseline_tournament_ms=min(ms[2]), baseline_tournament_ms_all=ms[2])
        hg, ht = min(ms[-2]), min(ms[-1])
        rows[-1].update(h2h_group_stage_ms=hg, h2h_tournament_ms=ht, h2h_group_stage_ms_all=ms[-2],
                        h2h_tournament_ms_all=ms[-1], h2h_group_stage_cost=hg / g - 1, h2h_tournament_cost=ht / t - 1)
        print(json.dumps(rows[-1]), flush=True)
    # the Champions League: its bracket with the real formats and with every tie one match, the league phase alone
    s_cl, fx_cl, hs_cl, as_cl, br_cl = champions_league(S)
    one = dict(br_cl, tie_format=np.zeros_like(br_cl["tie_format"]))
    K_cl, legs = len(br_cl["round"]), int((br_cl["tie_format"] == 2).sum())
    for R in (64,):
        lcall, lout, _lk = prepared_call(model, s_cl, fx_cl, hs_cl, as_cl, 36, None, R)
        fcall, fout, _fk = tournament_call(model, s_cl, fx_cl, hs_cl, as_cl, 36, None, br_cl, R)
        ocall, oout, _ok = tournament_call(model, s_cl, fx_cl, hs_cl, as_cl, 36, None, one, R)
        calls = [lcall, ocall, fcall]
        for _ in range(3):
            for c in calls:
                c()
        torch.cuda.synchronize()
        N = S * R
        assert all(int(o["invalid"].item()) == 0 for o in (lout, fout, oout))
        assert int(fout["decided"].sum()) == N * K_cl and int(fout["decided"].view(K_cl, 3)[:, 1].sum()) > 0
        ms = [[] for _ in calls]
        for _ in range(3):
            for c, m in zip(calls, ms):
                m.append(time_ms(c, a.reps))
        lg, o1, f2 = (min(m) for m in ms)
        rows.append({"workload": "champions league: 36-team league phase + 8 + 8 + 4 + 2 two-legged ties + final",
                     "model": model, "S": S, "R": R, "N": N, "F": len(hs_cl), "K": K_cl, "two_legged": legs,
                     "league_phase_ms": lg, "one_match_ms": o1, "formats_ms": f2, "league_phase_ms_all": ms[0],
                     "one_match_ms_all": ms[1], "formats_ms_all": ms[2],
                     "ps_per_sim_tie_one_match": (o1 - lg) * 1e9 / (N * K_cl),
                     "ps_per_sim_tie_formats": (f2 - lg) * 1e9 / (N * K_cl),
                     "ps_extra_per_sim_two_legged_tie": (f2 - o1) * 1e9 / (N * legs),
                     "decided_share": (fout["decided"].view(K_cl, 3).sum(0).double() / (N * K_cl)).tolist(),
                     "tournaments_per_s": N / (f2 * 1e-3)})
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
                                    "histograms": 48 * br["num_rounds"] * 8 + K * 8}}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
