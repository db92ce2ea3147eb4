"""Times season / group-stage simulation (bplx_simulate_table) on one GPU.

    python scripts/simulate_time.py [--samples 16384] [--reps 20] [--baseline-lib OLD/libbplx.so] [--out FILE.json]

Workloads (synthetic posterior draws, fixed seeds):
  league     20-team DixonColes league, F = 380 (a double round robin) and F = 190 (half a season), R = 64 and R = 1
  world cup  48-team group stage, 12 groups of four, 72 fixtures at neutral venues, NeutralWC draws of configs[5]'s shape
             (T = 220 model teams, Cf = 6), R = 64 and R = 1
With --baseline-lib, another build's bplx_simulate_table is timed on every workload, alternating with this build's, and
its counts are checked equal.  Every workload is also timed under the head-to-head ranking rule (bplx_simulate_table_ex,
no played matches), alternating with the goal-difference call in the same run: h2h_ms, h2h_cost = h2h_ms / ms - 1.
CUDA events around `--reps` calls after warm-up, best of three runs; a call is the whole entry point (count reset,
exponential-table pre-pass, simulation kernel), issued straight through the C ABI so that no host synchronisation sits
in the timed window.  Reports simulations/s and sampled scores/s, the GPU name and power limit read in the same run,
and the float64 oracle's CPU time on a few simulations of the league.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        import torch
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


def league(S, F):
    """20 teams, DixonColes draws; F = 380: every ordered pair once, F = 190: the first half of that list."""
    rng = np.random.default_rng(7)
    T = 20
    s = {"attack": rng.normal(0, 0.3, (S, T)).astype(np.float32), "defence": rng.normal(0, 0.3, (S, T)).astype(np.float32),
         "home_advantage": rng.normal(0.25, 0.05, S).astype(np.float32),
         "corr_coef": rng.uniform(-0.1, 0.1, S).astype(np.float32)}
    pairs = [(i, j) for i in range(T) for j in range(T) if i != j][:F]
    h, a = np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])
    fx = {"home_team": h.astype(np.uint16), "away_team": a.astype(np.uint16)}
    return "dixon_coles", s, fx, h.astype(np.uint8), a.astype(np.uint8), T, None


def world_cup(S):
    """48 of configs[5]'s 220 teams in 12 groups of four, each group a round robin at neutral venues."""
    from oracle import datasets

    s, _ = datasets.config_5(S=S, F=1)
    rng = np.random.default_rng(11)
    teams = rng.choice(220, 48, replace=False)
    group = np.repeat(np.arange(12), 4)
    hs, as_ = [], []
    for g in range(12):
        m = np.arange(4 * g, 4 * g + 4)
        for i in range(4):
            for j in range(i + 1, 4):
                hs.append(m[i])
                as_.append(m[j])
    hs, as_ = np.array(hs), np.array(as_)
    fx = {"home_team": teams[hs].astype(np.uint16), "away_team": teams[as_].astype(np.uint16),
          "home_conf": (teams[hs] % 6).astype(np.uint8), "away_conf": (teams[as_] % 6).astype(np.uint8),
          "neutral_venue": np.ones(len(hs), np.uint8)}
    return "neutral_wc", s, fx, hs.astype(np.uint8), as_.astype(np.uint8), 48, group.astype(np.uint8)


def device_table(T_tab, group, hs, as_):
    """A table of T_tab slots on the GPU, every team on zero, 3 points a win and 1 a draw, its histograms sized for the
    fixtures between slots hs and as_."""
    import torch

    from bpl_next_b200 import season

    zeros = torch.zeros(T_tab, dtype=torch.int32, device="cuda")
    tab = {"teams": range(T_tab), "group": group, "points_win": 3, "points_draw": 1}
    season._size_histograms(tab, hs, as_)
    tab.update(start_points=zeros, start_goals_for=zeros, start_goals_against=zeros,
               group=None if group is None else torch.from_numpy(group).cuda())
    return tab


def baseline_lib(path, names):
    """Another build's libbplx.so, its entry points ``names`` typed as this build's."""
    from bpl_next_b200 import _abi

    lib = C.CDLL(os.path.abspath(path))
    for name in names:
        getattr(lib, name).argtypes = getattr(_abi.lib(), name).argtypes
        getattr(lib, name).restype = getattr(_abi.lib(), name).restype
    return lib


def prepared_call(model, s, fx, hs, as_, T_tab, group, R, seed=1, lib=None, head_to_head=False):
    """The bplx_simulate_table call with every argument built once; returns (call, outputs, keep-alive).  ``lib``:
    another build's library (``baseline_lib``).  ``head_to_head``: bplx_simulate_table_ex under that ranking rule."""
    import torch

    from bpl_next_b200 import _abi, problem

    lib = _abi.lib() if lib is None else lib
    keep = []
    ptr = problem._device_ptr_fn(keep)
    dev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in s.items()}
    dfx = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in fx.items()}
    st = problem._samples_struct(model, dev, ptr)
    ft = problem._fixtures_struct(dfx, ptr)
    tab = device_table(T_tab, group, hs, as_)
    t = problem._table_struct(tab, ptr)
    d_hs, d_as = ptr(torch.from_numpy(hs).cuda()), ptr(torch.from_numpy(as_).cuda())
    pc = torch.empty((T_tab, t.num_positions), dtype=torch.int64, device="cuda")
    bc = torch.empty((T_tab, t.num_points_bins), dtype=torch.int64, device="cuda")
    inv = torch.empty(1, dtype=torch.int64, device="cuda")
    rk = _abi.Ranking(_abi.RANK_HEAD_TO_HEAD, None)
    if head_to_head:
        need = int(lib.bplx_simulate_table_ex_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t), C.byref(rk)))
    else:
        need = int(lib.bplx_simulate_workspace_bytes(C.byref(st), C.byref(ft), C.byref(t)))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    args = (C.byref(st), C.byref(ft), d_hs, d_as, C.byref(t)) + ((C.byref(rk),) if head_to_head else ()) + (
        15, R, seed, 0, ptr(pc), ptr(bc), None, None, ptr(inv), ptr(ws), ws.numel(), stream)
    fn = lib.bplx_simulate_table_ex if head_to_head else lib.bplx_simulate_table

    def call():
        rc = fn(*args)
        if rc != _abi.OK:
            raise _abi.BplxError(rc, lib.bplx_last_error().decode("utf-8", "replace"))

    return call, {"position_counts": pc, "points_counts": bc, "invalid": inv}, (keep, st, ft, t, dev, dfx, tab, ws, rk)


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
    ap.add_argument("--baseline-lib", default=None, help="another build's libbplx.so, timed on every workload")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from oracle import simulate as osim

    if not torch.cuda.is_available():
        raise SystemExit("simulate_time.py measures the GPU kernel and needs a CUDA device")
    S = a.samples
    rows = []
    base = None
    if a.baseline_lib:
        base = baseline_lib(a.baseline_lib, ("bplx_simulate_table", "bplx_simulate_workspace_bytes", "bplx_last_error"))
    for name, make in (("league F=380", lambda: league(S, 380)), ("league F=190", lambda: league(S, 190)),
                       ("world cup groups", lambda: world_cup(S))):
        model, s, fx, hs, as_, T_tab, group = make()
        for R in (64, 1):
            call, out, _keep = prepared_call(model, s, fx, hs, as_, T_tab, group, R)
            calls = [call]
            if base is not None:
                bcall, bout, _bk = prepared_call(model, s, fx, hs, as_, T_tab, group, R, lib=base)
                calls.append(bcall)
            hcall, hout, _hk = prepared_call(model, s, fx, hs, as_, T_tab, group, R, head_to_head=True)
            calls.append(hcall)
            for _ in range(3):
                for c in calls:
                    c()
            torch.cuda.synchronize()
            assert int(out["invalid"].item()) == 0 and int(hout["invalid"].item()) == 0
            assert torch.equal(out["points_counts"], hout["points_counts"])  # the rule moves positions only
            if base is not None:
                for k in ("position_counts", "points_counts", "invalid"):
                    assert torch.equal(out[k], bout[k]), k
            ms_all = [[] for _ in calls]
            for _ in range(3):  # alternate the builds
                for c, m in zip(calls, ms_all):
                    m.append(time_ms(c, a.reps))
            ms = min(ms_all[0])
            N, F = S * R, len(hs)
            rows.append({"workload": name, "model": model, "S": S, "R": R, "N": N, "F": F, "T_tab": T_tab,
                         "ms": ms, "ms_all": ms_all[0], "sims_per_s": N / (ms * 1e-3),
                         "scores_per_s": N * F / (ms * 1e-3)})
            if base is not None:
                rows[-1].update(baseline_ms=min(ms_all[1]), baseline_ms_all=ms_all[1])
            rows[-1].update(h2h_ms=min(ms_all[-1]), h2h_ms_all=ms_all[-1], h2h_cost=min(ms_all[-1]) / ms - 1,
                            h2h_changed_positions=int((out["position_counts"] != hout["position_counts"]).sum()))
            print(json.dumps(rows[-1]), flush=True)

    # the float64 oracle on the CPU: 2 draws x 64 simulations of the F = 380 league
    model, s, fx, hs, as_, T_tab, _ = league(2, 380)
    tab = {"start_points": np.zeros(T_tab, np.int32), "start_goals_for": np.zeros(T_tab, np.int32),
           "start_goals_against": np.zeros(T_tab, np.int32), "group": None, "points_win": 3, "points_draw": 1,
           "num_positions": T_tab, "num_points_bins": 3 * 38 + 1}
    t0 = time.perf_counter()
    osim.simulate(model, s, fx, hs, as_, tab, 15, 64, seed=1)
    t_or = time.perf_counter() - t0
    res = {"gpu": gpu_info(), "reps": a.reps, "workloads": rows,
           "oracle_cpu": {"sims": 128, "F": 380, "s": t_or, "sims_per_s": 128 / t_or}}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
