"""Times forecast uncertainty on BASELINE configs[4] (NeutralWC, T = 220, S = 16,384 synthetic draws, F = 10,000
fixtures) at max_goals 10 and 15 with predict_proba_posterior's default lines (totals 1.5, 2.5, 3.5; margins -1.5, 1.5:
K = 16 rows) and levels (0.05, 0.5, 0.95): the draws kernel with and without the [F K, S] matrix, the quantile kernel on
that matrix, the whole predictor method, and K3 (the averaged score grid) on the same inputs.

    python scripts/market_time.py [--reps 20] [--out FILE.json]

CUDA events around `--reps` calls after warm-up.  The matrix (10.5 GB) is far larger than L2, so every pass reaches HBM.
Each kernel's algorithmic bytes are set against the HBM floor at the data sheet's 7.7 TB/s (a computed floor, not a
measured peak).  The GPU's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
HBM_GBS = 7700.0  # NVIDIA HGX B200 data sheet, per GPU


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi gave nothing"


def time_ms(fn, reps):
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16384)
    ap.add_argument("--fixtures", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from bpl_next_b200 import NeutralDixonColesMatchPredictorWC
    from bpl_next_b200.problem import market_draws, market_names, row_quantiles, score_grid
    from oracle import datasets

    if not torch.cuda.is_available():
        raise SystemExit("market_time.py measures the GPU kernels and needs a CUDA device")
    S, F = a.samples, a.fixtures
    s, fx = datasets.config_5(S=S, F=F)
    ds = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fx.items()}
    tl, ml, lv = (1.5, 2.5, 3.5), (-1.5, 1.5), (0.05, 0.5, 0.95)
    K = len(market_names(tl, ml))
    mat = torch.empty((F * K, S), dtype=torch.float32, device="cuda")
    ws = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    p = NeutralDixonColesMatchPredictorWC()
    T, Cf = s["attack"].shape[1], s["confederation_strength"].shape[1]
    p.teams = [f"t{i}" for i in range(T)]
    p._teams_dict = {t: i for i, t in enumerate(p.teams)}
    p._conferences_dict = {f"c{i}": i for i in range(Cf)}
    for k, v in s.items():
        setattr(p, k, v)
    table_bytes = 4.0 * S * (6 * T + 2 * Cf + 4)

    out = {"gpu": gpu_info(), "S": S, "F": F, "K": K, "reps": a.reps, "hbm_floor_gbs": HBM_GBS,
           "hbm_floor_source": "NVIDIA HGX B200 data sheet, per GPU (computed, not measured)", "max_goals": {}}
    for G in (10, 15):
        def draws(want):
            return market_draws("neutral_wc", ds, dfx, G, tl, ml, want_matrix=want, draws=mat if want else None,
                                workspace=ws)

        def quant():
            return row_quantiles(mat, lv)

        def k3():
            return score_grid("neutral_wc", ds, dfx, G, workspace=ws)

        def method():
            return p.predict_proba_posterior(fx["home_team"], fx["away_team"], fx["home_conf"], fx["away_conf"],
                                             fx["neutral_venue"], max_goals=G)

        for _ in range(2):  # warm-up of every shape
            draws(True), draws(False), quant(), k3()
        method()
        torch.cuda.synchronize()
        mat_bytes = 4.0 * F * K * S
        g2 = (G + 1) ** 2
        rows = {"draws_with_matrix": {"ms": time_ms(lambda: draws(True), a.reps), "bytes": mat_bytes + table_bytes},
                "draws_no_matrix": {"ms": time_ms(lambda: draws(False), a.reps), "bytes": table_bytes + 16.0 * F * K},
                "quantiles": {"ms": time_ms(quant, a.reps), "bytes": mat_bytes + 8.0 * F * K * len(lv)},
                "k3_score_grid": {"ms": time_ms(k3, a.reps), "bytes": table_bytes + 4.0 * F * g2},
                "predict_proba_posterior": {"ms": time_ms(method, max(3, a.reps // 4)), "bytes": None}}
        for r in rows.values():
            if r["bytes"] is not None:
                r["floor_ms"] = r["bytes"] / (HBM_GBS * 1e9) * 1e3
                r["over_floor"] = r["ms"] / r["floor_ms"]
        # agreement in the same run: the outcome means against K3's averaged outcome
        _, st, inv = draws(False)
        _, outcome = k3()
        mean = st.cpu().numpy()[:, 0].reshape(F, K)
        rows["max_abs_outcome_mean_vs_k3"] = float(np.abs(mean[:, :3] - outcome.cpu().numpy()).max())
        rows["invalid"] = int(inv.item())
        out["max_goals"][str(G)] = rows
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
