"""Times the dynamic model's predictive calls on BASELINE configs[3]'s shape (T = 20, G = 30 gameweeks, 11,400 matches:
380 per gameweek) with S = 8,192 synthetic draws per gameweek (no fit needed):

* the segmented pointwise log-likelihood (one launch over all 30 gameweeks) + PSIS-LOO, against 30 per-gameweek
  NEUTRAL pointwise calls that produce the same matrix (checked bit for bit);
* the multi-gameweek posterior predictive check (every draw's 30 table rows in shared memory), against a one-gameweek
  NEUTRAL check of the same matches;
* the forecast at horizons 1 and 5.

    python scripts/dynamic_predict_time.py [--samples 8192] [--reps 10] [--out FILE.json]

CUDA events around `--reps` calls after warm-up; the GPU name, power limit and maximum SM clock are read in the same run.
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

from simulate_time import gpu_info, time_ms  # noqa: E402

SITES = ("attack", "defence", "home_attack", "away_attack", "home_defence", "away_defence")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from bpl_next_b200.problem import (dynamic_forecast, pointwise_loglik, pointwise_loglik_gameweeks,
                                       posterior_predictive, posterior_predictive_gameweeks, psis_loo)

    S, T, G = a.samples, 20, 30
    rng = np.random.default_rng(3)
    s = {k: torch.from_numpy(rng.normal(0, 0.3, (G, S, T)).astype(np.float32)).cuda() for k in SITES}
    s["corr_coef"] = torch.from_numpy(np.repeat(rng.uniform(-0.1, 0.05, (1, S)), G, 0).astype(np.float32)).cuda()
    pairs = [(h, w) for h in range(T) for w in range(T) if h != w]
    gw = np.repeat(np.arange(G), len(pairs))
    M = len(gw)
    obs = {"home_team": np.tile([p[0] for p in pairs], G).astype(np.uint16),
           "away_team": np.tile([p[1] for p in pairs], G).astype(np.uint16),
           "neutral_venue": np.zeros(M, np.uint8), "home_goals": rng.poisson(1.5, M).astype(np.uint8),
           "away_goals": rng.poisson(1.1, M).astype(np.uint8)}
    do = {k: torch.from_numpy(v).cuda() for k, v in obs.items()}
    res = {"gpu": gpu_info(), "S": S, "T": T, "G": G, "M": M, "reps": a.reps}

    # ---- pointwise log-likelihood + PSIS ----------------------------------------------------------------------------
    ll = torch.empty((M, S), dtype=torch.float32, device="cuda")
    ll_ref = torch.empty_like(ll)
    slabs = [{k: v[g] for k, v in s.items()} for g in range(G)]
    rows = [slice(g * len(pairs), (g + 1) * len(pairs)) for g in range(G)]
    do_g = [{k: v[r] for k, v in do.items()} for r in rows]

    def seg():
        pointwise_loglik_gameweeks("neutral", s, do, gw, loglik=ll)

    def per_gw():
        for g in range(G):
            pointwise_loglik("neutral", slabs[g], do_g[g], loglik=ll_ref[rows[g]])

    def loo():
        psis_loo(ll)

    for f in (seg, per_gw, loo):
        f()
    torch.cuda.synchronize()
    res["pointwise_bit_equal_to_per_gameweek_calls"] = bool(torch.equal(ll, ll_ref))
    res["pointwise_segmented_ms"] = time_ms(seg, a.reps)
    res["pointwise_30_neutral_calls_ms"] = time_ms(per_gw, a.reps)
    res["psis_ms"] = time_ms(loo, a.reps)
    res["pointwise_matrix_GB_per_s"] = M * S * 4 / (res["pointwise_segmented_ms"] * 1e-3) / 1e9

    # ---- posterior predictive check ---------------------------------------------------------------------------------
    def ppc_multi():
        posterior_predictive_gameweeks("neutral", s, do, gw, 15, 6, (3, 1), 1, 5)

    def ppc_one():
        posterior_predictive("neutral", slabs[G - 1], do, 15, 6, (3, 1), 1, 5)

    for f in (ppc_multi, ppc_one):
        f()
    res["ppc_multi_gameweek_ms"] = time_ms(ppc_multi, a.reps)
    res["ppc_one_gameweek_ms"] = time_ms(ppc_one, a.reps)
    res["ppc_scores_per_s"] = S * M / (res["ppc_multi_gameweek_ms"] * 1e-3)

    # ---- forecast ---------------------------------------------------------------------------------------------------
    att, dfn = s["attack"][G - 1].contiguous(), s["defence"][G - 1].contiguous()
    for h in (1, 5):
        dynamic_forecast(att, dfn, h, 1)
        res[f"forecast_h{h}_ms"] = time_ms(lambda: dynamic_forecast(att, dfn, h, 1), a.reps)
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
