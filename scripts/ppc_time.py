"""Times the posterior predictive kernel on BASELINE configs[2]'s data shape (NeutralWC, T = 220, M = 40,000 observed
matches) with S = 16,384 synthetic posterior draws, R = 1, max_goals 15: one replicate of all M matches per draw.

    python scripts/ppc_time.py [--samples 16384] [--reps 10] [--out FILE.json]

CUDA events around `--reps` calls after warm-up, with the raw scores off (statistics only) and on ([N, M, 2] uint8,
1.3 GB).  Reports the time per call and the sampled scores per second, scripts/simulate_time.py's league workload
(F = 380, R = 64) timed in the same run for reference, the float64 oracle's CPU rate on a slice, and the GPU name and
power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.dont_write_bytecode = True

from simulate_time import gpu_info, league, prepared_call, time_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--oracle-replicates", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from bpl_next_b200 import data as bdata
    from bpl_next_b200.problem import posterior_predictive
    from oracle import datasets
    from oracle import ppc as oppc

    if not torch.cuda.is_available():
        raise SystemExit("ppc_time.py measures the GPU kernel and needs a CUDA device")
    arr, _ = bdata.prepare("neutral_wc", datasets.config_3(), epsilon=0.1)
    S, M, T = a.samples, arr.num_matches, arr.num_teams
    s, _ = datasets.config_5(S=S, F=1)
    obs = {"home_team": arr.home_team, "away_team": arr.away_team, "neutral_venue": arr.neutral_venue,
           "home_conf": arr.home_conf, "away_conf": arr.away_conf, "home_goals": arr.home_goals,
           "away_goals": arr.away_goals}
    ds = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    do = {k: torch.from_numpy(np.ascontiguousarray(v).astype(np.uint16 if "team" in k else np.uint8)).cuda()
          for k, v in obs.items()}
    ws = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")

    def call(scores):
        return lambda: posterior_predictive("neutral_wc", ds, do, 15, 6, (3, 1), 1, 1, want_scores=scores, workspace=ws)

    for _ in range(2):  # warm-up of both shapes
        call(False)(), call(True)()
    torch.cuda.synchronize()
    out = call(True)()
    noraw = call(False)()
    assert int(out["invalid"].item()) == 0
    assert torch.equal(out["team_points"], noraw["team_points"])
    rows = {}
    for name, scores in (("statistics_only", False), ("with_raw_scores", True)):
        ms_all = [time_ms(call(scores), a.reps) for _ in range(3)]
        ms = min(ms_all)
        rows[name] = {"ms": ms, "ms_all": ms_all, "scores_per_s": S * M / (ms * 1e-3)}
        print(json.dumps({name: rows[name]}), flush=True)

    # the season simulation's league workload, for reference
    model, ls, fx, hs, as_, T_tab, group = league(S, 380)
    scall, sout, _keep = prepared_call(model, ls, fx, hs, as_, T_tab, group, 64)
    for _ in range(3):
        scall()
    torch.cuda.synchronize()
    sms = min(time_ms(scall, a.reps) for _ in range(3))
    sim = {"workload": "league F=380", "S": S, "R": 64, "ms": sms, "scores_per_s": S * 64 * 380 / (sms * 1e-3)}

    # the float64 oracle on the CPU: a few replicates of the first 4,000 matches, checked against the kernel's scores
    n = min(4000, M)
    sub = {k: v[:n] for k, v in obs.items()}
    s_or = {k: v[:a.oracle_replicates] for k, v in s.items()}
    t0 = time.perf_counter()
    home, away, margin, valid = oppc.replicate("neutral_wc", s_or, sub, 15, 1, 1)
    t_or = time.perf_counter() - t0
    ksc = out["scores"][:a.oracle_replicates, :n].cpu().numpy().astype(np.int64)
    diff = (ksc[..., 0] != home) | (ksc[..., 1] != away)
    res = {"gpu": gpu_info(), "S": S, "M": M, "T": T, "R": 1, "max_goals": 15, "score_bins": 6, "reps": a.reps,
           "kernels": rows, "simulate_table_reference": sim,
           "oracle_cpu": {"replicates": a.oracle_replicates, "matches": n, "s": t_or,
                          "scores_per_s": a.oracle_replicates * n / t_or},
           "oracle_score_mismatches": int(diff.sum()), "oracle_mismatches_off_boundary": int((diff & (margin >= 1e-5)).sum())}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
