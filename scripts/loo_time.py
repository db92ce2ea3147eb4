"""Times the model-comparison kernels on BASELINE configs[2] (NeutralWC, T = 220, M = 40,000) with S = 16,384 synthetic
posterior draws: the pointwise log-likelihood kernel with and without the [M, S] matrix, and PSIS-LOO on that matrix.

    python scripts/loo_time.py [--samples 16384] [--reps 20] [--out FILE.json]

CUDA events around `--reps` launches after warm-up.  The matrix (2.6 GB) is larger than L2, so every pass reaches HBM.
Prints the algorithmic bytes of each kernel and its share of the HBM floor, against the same peak bench.py uses (the
measured MEASURED_PEAKS.json when present, else 6,650 GB/s), the GPU name and power limit read in the same run, and the
float64 oracle's CPU time on 500 matches.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback 6650 GB/s (bench.py's default)"


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        import torch
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--oracle-matches", type=int, default=500)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from bpl_next_b200 import data as bdata
    from bpl_next_b200.problem import pointwise_loglik, psis_loo
    from oracle import datasets, psis

    if not torch.cuda.is_available():
        raise SystemExit("loo_time.py measures the GPU kernels and needs a CUDA device")
    arr, _ = bdata.prepare("neutral_wc", datasets.config_3(), epsilon=0.1)
    S, M = a.samples, arr.num_matches
    s, _ = datasets.config_5(S=S, F=1)
    obs = {"home_team": arr.home_team, "away_team": arr.away_team, "neutral_venue": arr.neutral_venue,
           "home_conf": arr.home_conf, "away_conf": arr.away_conf, "home_goals": arr.home_goals,
           "away_goals": arr.away_goals}
    ds = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    do = {k: torch.from_numpy(np.ascontiguousarray(v).astype(np.uint16 if "team" in k else np.uint8)).cuda()
          for k, v in obs.items()}
    mat = torch.empty((M, S), dtype=torch.float32, device="cuda")
    ws = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")

    def pw(want):
        return pointwise_loglik("neutral_wc", ds, do, want_matrix=want, loglik=mat if want else None, workspace=ws)

    def ps():
        return psis_loo(mat, 1.0)

    for _ in range(3):  # warm-up of every shape
        pw(True), pw(False), ps()
    torch.cuda.synchronize()
    t_mat, t_nomat, t_psis = time_ms(lambda: pw(True), a.reps), time_ms(lambda: pw(False), a.reps), time_ms(ps, a.reps)

    peak, src = hbm_peak()
    mat_bytes = 4.0 * M * S
    rows = {
        "pointwise_with_matrix": {"ms": t_mat, "bytes": mat_bytes + 32.0 * M},
        "pointwise_no_matrix": {"ms": t_nomat, "bytes": 32.0 * M},
        "psis_loo": {"ms": t_psis, "bytes": mat_bytes + 16.0 * M},
    }
    for r in rows.values():
        r["gbs"] = r["bytes"] / (r["ms"] * 1e-3) / 1e9
        r["floor_ms"] = r["bytes"] / (peak * 1e9) * 1e3
        r["frac_of_hbm_floor"] = r["floor_ms"] / r["ms"]

    # the float64 oracle on the CPU, a slice of the same problem
    n = min(a.oracle_matches, M)
    ll = mat[:n].cpu().numpy().T.astype(np.float64)
    t0 = time.perf_counter()
    ll_o = psis.pointwise_loglik("neutral_wc", s, arr.home_team[:n], arr.away_team[:n], arr.home_goals[:n],
                                 arr.away_goals[:n], home_conf=arr.home_conf[:n], away_conf=arr.away_conf[:n],
                                 neutral_venue=arr.neutral_venue[:n])
    e_o, k_o = psis.loo_pointwise(ll_o)
    t_oracle = time.perf_counter() - t0
    e, k = psis_loo(mat[:n], 1.0)
    e_o, k_o = psis.loo_pointwise(ll)  # PSIS of the oracle on the kernel's own float32 matrix
    e, k = e.cpu().numpy(), k.cpu().numpy()
    fe, fk = np.isfinite(e_o), np.isfinite(k_o)  # (matches with a -inf draw: NaN / inf in both)
    out = {"gpu": gpu_info(), "S": S, "M": M, "tail_draws": psis.tail_length(S), "reps": a.reps,
           "hbm_peak_gbs": peak, "hbm_peak_source": src, "kernels": rows,
           "oracle_cpu_s_on_%d_matches" % n: t_oracle,
           "neg_inf_entries_agree": bool((np.isneginf(ll) == np.isneginf(ll_o)).all()),
           "max_abs_ll_err_vs_oracle": float(np.abs(ll - ll_o)[np.isfinite(ll_o)].max()),
           "max_rel_elpd_err_vs_oracle": float(np.abs(e[fe] / e_o[fe] - 1).max()) if fe.any() else None,
           "max_khat_err_vs_oracle": float(np.abs(k[fk] - k_o[fk]).max()) if fk.any() else None}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
