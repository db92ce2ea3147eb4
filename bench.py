#!/usr/bin/env python
"""bench.py -- log-density+gradient match-evaluations per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch: one `bplx_logdensity_fwdbwd` call for all the chains of
this GPU; the timed windows of `value` and of `e2e` are exactly K steps each.  The workload is the configuration
the metric is quoted on, BASELINE.json configs[2] (NeutralDixonColesMatchPredictorWC, 220 teams, 40,000 weighted
matches, 32,768 chains): at N GPUs the 32,768 chains are partitioned over the ranks (STRONG scaling, chains are independent: no data-path collective).
`value` times the kernel with inputs resident in HBM (CUDA graph of K launches over rotating buffer sets larger
than L2, CUDA events on the launch stream, max over ranks); `e2e` goes through the host-buffer C-ABI call with
pinned host arrays, copies inside the timed region.  Two sub-records are timed on all ranks: the configs[4]
predictive grid with posterior samples sharded S/N and the NCCL all-reduce inside the CUDA-event region, and a
chain-sharded configs[2] `fit` with its R-hat / ESS moment all-reduce and summary gather.
`--impl reference` times the CPU restatement of the reference (oracle/closed_form.py, float32, all host
threads) on bounded samples of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree, which may be read-only

L2_BYTES = 126e6
FLOPS_PER_EVAL = {"dixon_coles": 26, "extended": 30, "neutral": 40, "neutral_wc": 46, "dynamic": 40}  # SURVEY.md 8(d)
METRIC = "logdensity_grad_match_evals_per_s"
UNIT = "match-evals/s"


# ------------------------------------------------------------------------------------------------
# workloads (synthetic; oracle/datasets.py only generates inputs here)
# ------------------------------------------------------------------------------------------------
def workload(name):
    from bpl_next_b200 import data as bdata
    from oracle import datasets

    if name == "cfg2":
        arr, _ = bdata.prepare("extended", datasets.config_2(), epsilon=0.01)
        desc = "configs[1]: ExtendedDixonColes T=20, 5 seasons M=1900, K=3 covariates, eps=0.01"
        return arr, 4096, desc
    if name == "cfg3":
        arr, _ = bdata.prepare("neutral_wc", datasets.config_3(), epsilon=0.1)
        desc = "configs[2]: NeutralDixonColesMatchPredictorWC T=220, M=40000 weighted, Cf=6"
        return arr, 32768, desc
    if name == "cfg4":
        arr, _ = bdata.prepare("dynamic", datasets.config_4())
        desc = "configs[3]: DynamicDixonColes T=20, 30 seasons M=11400, G=30 (intended random walk)"
        return arr, 8192, desc
    if name == "cfg1":
        arr, _ = bdata.prepare("dixon_coles", datasets.dummy_data())
        return arr, 4096, "configs[0] data: DixonColes T=20 M=380"
    raise ValueError(name)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written) + FFMA / smem peaks measured now."""
    out = {"hbm_gbs": 6650.0, "hbm_source": "fallback"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            out["hbm_gbs"] = float(json.load(f)["hbm_gbs"])
        out["hbm_source"] = "measured (MEASURED_PEAKS.json)"
    lib = ctypes.CDLL(os.path.join(ROOT, "bpl_next_b200", "lib", "libbplx_bench.so"))
    lib.bplxbench_fp32_peak.restype = ctypes.c_double
    lib.bplxbench_smem_peak.restype = ctypes.c_double
    out["fp32_tflops"] = float(lib.bplxbench_fp32_peak(2000, 5))
    out["smem_tbs"] = float(lib.bplxbench_smem_peak(2000, 5))
    return out


def shard(n, rank, world):
    base, extra = divmod(n, world)
    return rank * base + min(rank, extra), base + (1 if rank < extra else 0)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def parity_sample(arr, theta_dc, lp, grad, cc, nsample=8, seed=0):
    """`nsample` chains of a [D, C] batch the kernel has just evaluated, against the float64 oracle (test infrastructure
    used as the checker): max relative lp error, max gradient error scaled by the chain's largest gradient entry."""
    from oracle import models as om
    from tests import helpers as H

    C = theta_dc.shape[1]
    idx = np.unique(np.concatenate([[0, C - 1], np.random.default_rng(seed).integers(0, C, nsample)]))
    th = theta_dc[:, idx].T.contiguous().cpu().numpy().astype(np.float64)
    lp_o, g_o, cc_o = om.log_density_and_grad(H.to_oracle(arr), th)
    lp_k = lp[idx].cpu().numpy().astype(np.float64)
    g_k = grad[:, idx].T.cpu().numpy().astype(np.float64)
    ok = np.isfinite(lp_o)
    e_lp = float(np.max(np.abs(lp_k[ok] - lp_o[ok]) / np.abs(lp_o[ok]))) if ok.any() else float("nan")
    e_g = float(np.max(np.abs(g_k[ok] - g_o[ok]) / np.abs(g_o[ok]).max(axis=1, keepdims=True))) if ok.any() else float("nan")
    e_c = float(np.max(np.abs(cc[idx].cpu().numpy()[ok] - cc_o[ok]))) if ok.any() else float("nan")
    return {"chains_checked": int(ok.sum()), "lp_rel": e_lp, "grad_scaled": e_g, "corr_coef_abs": e_c,
            "tolerance": {"lp_rel": 1e-5, "grad_scaled": 1e-4}, "ok": bool(e_lp < 1e-5 and e_g < 1e-4)}


def time_logdensity(problem, C, steps, warmup, radius, seed, use_graph=True, target_s=1.0, arr=None, pad_rows=False):
    """Device time of a K-step region (ms): of one region when target_s is 0, else the median over repetitions for
    target_s seconds; inputs rotate through buffer sets whose total size exceeds the L2 whatever K is."""
    import torch

    from bpl_next_b200 import _abi

    D = problem.D
    set_bytes = 2 * C * D * 4
    nb = max(2, int(math.ceil(1.5 * L2_BYTES / set_bytes)))
    g = torch.Generator(device="cuda").manual_seed(seed)
    # row pitch of the [D, C] arrays (the C ABI's `ld` argument): dense by default; --pad-rows adds one 128-byte line to a
    # pitch that is a multiple of 4 KB (measured: no difference on B200 for K1, K1d or the NUTS step)
    ld = C + 32 if (pad_rows and (C * 4) % 4096 == 0) else C
    thetas = [((torch.rand((D, ld), generator=g, device="cuda", dtype=torch.float32) * 2 - 1) * radius)[:, :C] for _ in range(nb)]
    grads = [torch.empty((D, ld), device="cuda", dtype=torch.float32)[:, :C] for _ in range(nb)]
    lps = [torch.empty(C, device="cuda", dtype=torch.float32) for _ in range(nb)]
    ccs = [torch.empty(C, device="cuda", dtype=torch.float32) for _ in range(nb)]
    problem.workspace(C)
    stream = torch.cuda.Stream()
    lib = _abi.lib()

    def launch(k):
        i = k % nb
        problem.logdensity(thetas[i], chain_minor=True, lp=lps[i], grad=grads[i], corr_coef=ccs[i], stream=stream)

    parity = None
    with torch.cuda.stream(stream):
        for k in range(max(warmup, nb)):
            launch(k)
        stream.synchronize()
        if arr is not None:  # the same launch geometry as the timed region, checked against the oracle
            parity = parity_sample(arr, thetas[0], lps[0], grads[0], ccs[0])
        graph = None
        l0 = lib.bplx_launch_count()
        if use_graph:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                for k in range(steps):
                    launch(k)
            launches = int(lib.bplx_launch_count() - l0)

        def region():
            if graph is not None:
                graph.replay()
            else:
                for k in range(steps):
                    launch(k)

        region()  # warm the graph / caches once
        stream.synchronize()
        if not use_graph:
            launches = int(lib.bplx_launch_count() - l0)
        times = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start = time.perf_counter()
        while True:
            e0.record(stream)
            region()
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
            if time.perf_counter() - t_start > target_s or len(times) >= 400:
                break
    finite = bool(torch.isfinite(lps[0]).all().item())
    last = (steps - 1) % nb  # the buffer set the last step of the region wrote
    return {"ms": float(np.median(times)), "reps": len(times), "nb": nb, "set_bytes": set_bytes, "finite": finite, "ld": ld,
            "launches": launches, "parity": parity, "last": (lps[last], grads[last], ccs[last])}


DUMP_GRAD_BYTES = 48 << 20


def dump_outputs(out_dir, lp, grad, corr_coef, suffix=""):
    """The outputs of one log-density call as float32 .npy files: lp [C], corr_coef [C] and grad [D, C].  A gradient
    larger than DUMP_GRAD_BYTES is written for a sample of chains only: the columns np.random.default_rng(0) draws
    without replacement, in ascending order, so that runs with the same arguments write the same chains."""
    import torch

    D, C = grad.shape
    n = min(C, DUMP_GRAD_BYTES // (4 * D))
    if n < C:
        cols = np.sort(np.random.default_rng(0).choice(C, n, replace=False))
        grad = grad[:, torch.from_numpy(cols).to(grad.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("lp", lp), ("grad", grad), ("corr_coef", corr_coef)):
        np.save(os.path.join(out_dir, name + suffix + ".npy"), t.cpu().numpy().astype(np.float32))


def time_e2e(problem, C, steps, warmup, radius, seed):
    """Host-buffer entry point: pinned numpy in, pinned numpy out, copies inside the timed region."""
    import torch

    D = problem.D
    rng = np.random.default_rng(seed)
    nb = 2 if C * D * 4 > 64e6 else 4
    th = [torch.empty((C, D), dtype=torch.float32).pin_memory() for _ in range(nb)]
    for t in th:
        t.numpy()[:] = rng.uniform(-radius, radius, (C, D)).astype(np.float32)
    lp = torch.empty(C, dtype=torch.float32).pin_memory()
    gr = torch.empty((C, D), dtype=torch.float32).pin_memory()
    cc = torch.empty(C, dtype=torch.float32).pin_memory()
    for k in range(max(warmup, 3)):
        problem.logdensity_host(th[k % nb].numpy(), lp=lp.numpy(), grad=gr.numpy(), corr_coef=cc.numpy())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        problem.logdensity_host(th[k % nb].numpy(), lp=lp.numpy(), grad=gr.numpy(), corr_coef=cc.numpy())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, C * D * 4, C * D * 4 + 2 * C * 4


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle/ as the thing timed: only here)
# ------------------------------------------------------------------------------------------------
def cpu_evaluator(arr):
    """(callable theta -> (lp, grad, cc), description).  Static models: float32 closed-form gradient (SURVEY
    Appendix B, what a fused XLA:CPU value_and_grad amounts to); dynamic: float32 autograd of the restatement."""
    import torch

    from oracle import closed_form as cf, models as om
    from tests import helpers as H

    d = H.to_oracle(arr)
    torch.set_num_threads(os.cpu_count() or 1)
    if arr.model == "dynamic":
        return (lambda th: om.log_density_and_grad(d, th, dtype=torch.float32)), \
            "oracle/models.py float32 value + autograd gradient"
    return cf.ClosedForm(d, torch.float32), "oracle/closed_form.py float32 value + closed-form gradient (SURVEY Appendix B)"


def cpu_port(arr, C_total, C_sample, min_seconds, radius, seed, max_calls=1000):
    """The restatement on all host threads, chains in RAM-sized blocks; returns evals/s and details."""
    import torch

    from oracle import models as om
    from tests import helpers as H

    f, how = cpu_evaluator(arr)
    D = om.num_params(arr.model, arr.num_teams, arr.num_covariates, arr.num_conferences, arr.num_gameweeks)
    theta = np.random.default_rng(seed).uniform(-radius, radius, (C_sample, D)).astype(np.float32)
    f(theta)  # warm-up
    calls, t0 = 0, time.perf_counter()
    per_call = []
    while True:
        t1 = time.perf_counter()
        f(theta)
        per_call.append(time.perf_counter() - t1)
        calls += 1
        if time.perf_counter() - t0 >= min_seconds or calls >= max_calls:
            break
    dt = time.perf_counter() - t0
    out = {"value": C_sample * arr.num_matches * calls / dt, "unit": UNIT, "cores": torch.get_num_threads(),
           "kind": "port", "per_call_s": float(np.median(per_call)), "calls": calls,
           "sample": f"blocks of {C_sample} chains x {arr.num_matches} matches (of the workload's {C_total} chains), "
                     f"{calls} blocks in {dt:.1f} s, {how}; restatement of the reference, not its binary "
                     "(jax / numpyro are not installable in this image)"}
    if arr.model != "dynamic":  # second figure: autograd of the line-by-line restatement (round 1's baseline)
        d = H.to_oracle(arr)
        th = theta[:min(C_sample, 128)]
        om.log_density_and_grad(d, th, dtype=torch.float32)
        t1 = time.perf_counter()
        n = 0
        while time.perf_counter() - t1 < 3.0:
            om.log_density_and_grad(d, th, dtype=torch.float32)
            n += 1
        out["autograd_value"] = len(th) * arr.num_matches * n / (time.perf_counter() - t1)
    return out


def run_reference(args, rank, world):
    """Reference arm: the CPU restatement timed on the host cores (rank 0 only)."""
    if rank != 0:
        return
    import torch

    from oracle import models as om

    arr, C, desc = workload(args.workload)
    if args.chains:
        C = args.chains
    C_sample = args.cpu_chains
    f, how = cpu_evaluator(arr)
    D = om.num_params(arr.model, arr.num_teams, arr.num_covariates, arr.num_conferences, arr.num_gameweeks)
    theta = np.random.default_rng(args.seed + 1).uniform(-args.radius, args.radius, (C_sample, D)).astype(np.float32)
    for _ in range(max(min(args.warmup, 3), 1)):
        f(theta)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        f(theta)
    dt = time.perf_counter() - t0
    value = C_sample * arr.num_matches * args.steps / dt
    sample = (f"each step = one block of {C_sample} chains x {arr.num_matches} matches (bounded sample of the workload's "
              f"{C} chains), {how}, all host threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc + f", {C} chains in total", "chains_total": C, "matches": arr.num_matches,
                       "teams": arr.num_teams, "params": D, "theta": f"U(-{args.radius},{args.radius})"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# sub-records timed on ALL ranks (north_star's multi-GPU splits)
# ------------------------------------------------------------------------------------------------
def sub_grid(rank, world, reps=5):
    """configs[4]: S=16,384 posterior samples x F=10,000 fixtures x 11x11, samples sharded S/N; the all-reduce of
    [F,11,11] + [F,3] is INSIDE the CUDA-event region (compute and exchange also timed separately)."""
    import torch
    import torch.distributed as dist

    from bpl_next_b200 import parallel
    from oracle import datasets

    s, fx = datasets.config_5()
    S, F = s["attack"].shape[0], len(fx["home_team"])
    s0, sn = shard(S, rank, world)
    ds = {k: torch.from_numpy(np.ascontiguousarray(v[s0:s0 + sn])).cuda() for k, v in s.items()}
    dfx = {k: torch.from_numpy(v).cuda() for k, v in fx.items()}
    sg = parallel.ShardedScoreGrid("neutral_wc", ds, dfx, 10, num_samples_total=S)
    for _ in range(3):
        sg.run()
    torch.cuda.synchronize()
    tot, comp, exch = [], [], []
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = sg.run(timed=True)
        tot.append(t[0]); comp.append(t[1]); exch.append(t[2])
    grid, outc = sg.grid, sg.outcome
    t = torch.tensor([np.median(tot), np.median(comp), np.median(exch)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_c, ms_x = (float(x) for x in t.tolist())
    flops = S * F * (2 * 121 + 2 * 2 * 11 + 12)  # SURVEY.md 8(d), whole job
    rec = {"workload": f"configs[4]: predict grid S={S} x F={F} x 11x11, samples sharded {S}/{world} per GPU",
           "metric": "score_grid_ms", "value": ms, "unit": "ms (compute + all-reduce, max over ranks)",
           "compute_ms": ms_c, "allreduce_ms": ms_x, "allreduce_frac": ms_x / ms if ms > 0 else None,
           "allreduce_bytes": int(grid.numel() * 4 + outc.numel() * 4), "exchange": sg.exchange_kind,
           "sample_fixture_pairs_per_s": S * F / (ms * 1e-3), "n_gpus": world,
           "outcome_sum_err": float((outc.sum(dim=1) - 1).abs().max().item())}
    # parity on 64 random fixtures against the oracle (full S): rank 0 only, the all-reduced grid
    if rank == 0:
        from oracle import predict as op
        idx = np.random.default_rng(7).choice(F, 64, replace=False)
        g_ref, _, _ = op.predict_score_grid_proba("neutral_wc", s, fx["home_team"][idx], fx["away_team"][idx], 10,
                                                  home_conf=fx["home_conf"][idx], away_conf=fx["away_conf"][idx],
                                                  neutral_venue=fx["neutral_venue"][idx])
        rec["parity_max_abs_err"] = float(np.abs(grid[torch.from_numpy(idx).cuda()].cpu().numpy() - g_ref).max())
        rec["parity_tolerance"] = 1e-6
    return rec, flops


def sub_fit(rank, world, args):
    """configs[2] `fit`, chains sharded over the ranks: no collective while sampling; the split-R-hat / ESS moments
    are all-reduced and the posterior summary gathered at the end (both inside the wall-clock)."""
    import torch
    import torch.distributed as dist

    from bpl_next_b200 import NeutralDixonColesMatchPredictorWC
    from oracle import datasets

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    m = NeutralDixonColesMatchPredictorWC()
    out = m.fit_streaming(datasets.config_3(), epsilon=0.1, num_warmup=args.fit_warmup, num_samples=args.fit_samples,
                          num_chains=args.fit_chains, thin=args.fit_thin, max_tree_depth=args.fit_tree_depth,
                          max_launches=args.fit_max_launches or None)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    rec = {"workload": f"configs[2]: NeutralDixonColesMatchPredictorWC.fit T=220 M=40000, {args.fit_chains} chains sharded "
                       f"over {world} GPU(s), {args.fit_warmup} warmup + {args.fit_samples} draws (thin {args.fit_thin}), "
                       f"max_tree_depth {args.fit_tree_depth}",
           "metric": "ess_per_s", "value": out["ess_min"] / wall, "unit": "min-over-parameters bulk ESS / s (whole fit)",
           "fit_wall_s": wall, "n_gpus": world}
    rec.update({k: v for k, v in out.items()})
    return rec


# ------------------------------------------------------------------------------------------------
# extras: other configs on one GPU (rank 0, N=1 only)
# ------------------------------------------------------------------------------------------------
def extras(args, pk):
    import torch

    from bpl_next_b200 import Problem, score_grid
    from oracle import datasets

    out = []
    # configs[1]: Extended, 4,096 chains on one GPU -- init_to_uniform(2) inputs and typical-set inputs
    arr, C, desc = workload("cfg2")
    p = Problem(arr)
    for radius, note in ((args.radius, ""), (0.2, " (typical-set inputs: clip-free forms)")):
        r = time_logdensity(p, C, 50, 5, radius, args.seed + 9, use_graph=True, target_s=0.5, arr=arr)
        evals = C * arr.num_matches * 50 / (r["ms"] * 1e-3)
        out.append({"workload": desc + f", {C} chains on 1 GPU, theta U(-{radius},{radius}){note}",
                    "metric": METRIC, "value": evals, "unit": UNIT, "ms_per_call": r["ms"] / 50, "finite": r["finite"],
                    "parity_max_err": r["parity"],
                    "fp32_frac": FLOPS_PER_EVAL[arr.model] * evals / 1e12 / pk["fp32_tflops"]})
    p.close()
    del p
    # the few-chain ("streaming") regime on configs[2] data
    arr, C, desc = workload("cfg3")
    p = Problem(arr)
    st = p.stats()
    plan_bytes = 8 * (st["entries1_padded"] + st["entries2_padded"]) + 16 * 2600
    for Cs in (1, 32):
        r = time_logdensity(p, Cs, 20, 3, args.radius, args.seed + 5, use_graph=True, target_s=0.3, arr=arr)
        ms1 = r["ms"] / 20
        out.append({"workload": desc + f", {Cs} chain(s): few-chain (streaming) regime", "metric": METRIC,
                    "value": Cs * arr.num_matches / (ms1 * 1e-3), "unit": UNIT, "ms_per_call": ms1, "finite": r["finite"],
                    "parity_max_err": r["parity"],
                    "match_bytes_gbs": 13.0 * arr.num_matches / (ms1 * 1e-3) / 1e9,
                    "plan_stream_gbs": plan_bytes / (ms1 * 1e-3) / 1e9, "hbm_peak_gbs": pk["hbm_gbs"]})
    p.close()
    del p
    torch.cuda.empty_cache()
    # configs[3]: Dynamic, 8,192 chains (theta radius 0.5: a 30-step walk of U(-2,2) steps overflows float32 rates)
    arr, C, desc = workload("cfg4")
    p = Problem(arr)
    r = time_logdensity(p, C, 5, 3, 0.5, args.seed + 4, use_graph=False, target_s=0.5, arr=arr)
    evals = C * arr.num_matches * 5 / (r["ms"] * 1e-3)
    out.append({"workload": desc + f", {C} chains on 1 GPU, theta U(-0.5,0.5)", "metric": METRIC, "value": evals,
                "unit": UNIT, "ms_per_call": r["ms"] / 5, "finite": r["finite"], "plan": p.stats(),
                "parity_max_err": r["parity"],
                "fp32_frac": FLOPS_PER_EVAL["dynamic"] * evals / 1e12 / pk["fp32_tflops"],
                "hbm_frac": (8.0 * p.D * C) / (r["ms"] / 5 * 1e-3) / 1e9 / pk["hbm_gbs"]})
    p.close()
    del p
    torch.cuda.empty_cache()
    # ESS/s of whole fits (warm-up included): configs[0] at 1 and 1,024 chains, configs[1] at 4,096 chains
    try:
        from bpl_next_b200 import DixonColesMatchPredictor, ExtendedDixonColesMatchPredictor, diagnostics as dg
        jobs = [("configs[0]: DixonColesMatchPredictor.fit T=20 M=380", DixonColesMatchPredictor, datasets.dummy_data(), {},
                 1, 500, 1000, 380),
                ("configs[0]: DixonColesMatchPredictor.fit T=20 M=380", DixonColesMatchPredictor, datasets.dummy_data(), {},
                 1024, 500, 250, 380),
                ("configs[1]: ExtendedDixonColesMatchPredictor.fit T=20 M=1900 K=3", ExtendedDixonColesMatchPredictor,
                 datasets.config_2(), {"epsilon": 0.01}, 4096, 300, 100, 1900)]
        for name, cls, td, kw, chains, nw, ns, M in jobs:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = cls().fit(td, num_warmup=nw, num_samples=ns, mcmc_kwargs={"num_chains": chains}, **kw)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            run = m.nuts_run
            ess = dg.effective_sample_size(run.samples)
            rhat = dg.split_rhat(run.samples) if ns >= 4 else None
            out.append({"workload": f"{name}, {chains} chain(s), {nw} warmup + {ns} draws",
                        "metric": "ess_per_s", "value": float(ess.min().item()) / wall, "unit": "min-over-parameters bulk ESS / s",
                        "fit_wall_s": wall, "ess_min": float(ess.min().item()), "ess_median": float(ess.median().item()),
                        "rhat_max": None if rhat is None else float(rhat.max().item()),
                        "logdensity_launches": int(run.launches), "leapfrogs_total": int(run.num_leapfrog.sum()),
                        "divergences": int(run.num_divergent.sum()),
                        "match_evals_per_s_inside_fit": float(run.num_leapfrog.sum()) * M / wall})
            del m, run
            torch.cuda.empty_cache()
    except Exception as e:  # never lose the main line
        out.append({"workload": "fits", "error": repr(e)})
    # the reference's default max_goals=15 (16x16 cells, two 8x16 tiles per fixture) on the configs[4] inputs
    try:
        s, fx = datasets.config_5()
        ds = {k: torch.from_numpy(v).cuda() for k, v in s.items()}
        dfx = {k: torch.from_numpy(v).cuda() for k, v in fx.items()}
        S, F = s["attack"].shape[0], len(fx["home_team"])
        ws = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
        for _ in range(2):
            score_grid("neutral_wc", ds, dfx, 15, workspace=ws)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for _ in range(3):
            e0.record()
            score_grid("neutral_wc", ds, dfx, 15, workspace=ws)
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = float(np.median(ts))
        flops = S * F * (2 * 256 + 2 * 2 * 16 + 12)
        out.append({"workload": f"configs[4] inputs at the reference's default max_goals=15 (16x16) on 1 GPU",
                    "metric": "score_grid_ms", "value": ms, "unit": "ms",
                    "fp32_frac": flops / (ms * 1e-3) / 1e12 / pk["fp32_tflops"]})
    except Exception as e:
        out.append({"workload": "grid max_goals=15", "error": repr(e)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="bplx", choices=["bplx", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg1", "cfg2", "cfg3", "cfg4"])
    ap.add_argument("--chains", type=int, default=0, help="chains IN TOTAL over all GPUs (default: the workload's)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the chains are partitioned over the GPUs; weak: every GPU gets all of them")
    ap.add_argument("--radius", type=float, default=2.0, help="theta ~ U(-radius, radius) (numpyro init_to_uniform)")
    ap.add_argument("--seed", type=int, default=1002)
    ap.add_argument("--cpu-chains", type=int, default=256, help="chains per block of the CPU restatement")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--pad-rows", action="store_true", help="row pitch of theta / grad C + 32 floats instead of C")
    ap.add_argument("--fit-chains", type=int, default=32768)
    ap.add_argument("--fit-warmup", type=int, default=100)
    ap.add_argument("--fit-samples", type=int, default=50)
    ap.add_argument("--fit-thin", type=int, default=5)
    ap.add_argument("--fit-tree-depth", type=int, default=5,
                    help="max_tree_depth of the fit sub-record (numpyro's default is 10; 5 bounds the bench's wall time: "
                         "before the mass matrix is adapted every transition of this 1,339-parameter posterior runs to the "
                         "cap, so the sub-record is a timing of the sharded fit path, not a converged posterior -- see rhat_max)")
    ap.add_argument("--fit-max-launches", type=int, default=0, help="cap on log-density launches of the fit sub-record (0: none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write lp, grad and corr_coef of the last one as DIR/<name>.npy (float32; "
                         "grad [D, chains] for a fixed sample of chains when it is larger than 48 MiB; one set per rank, "
                         "suffixed _rank<r>, when there are several)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from bpl_next_b200 import Problem, _abi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (bpl_next_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    arr, C_total, desc = workload(args.workload)
    if args.chains:
        C_total = args.chains
    C = shard(C_total, rank, world)[1] if args.scaling == "strong" else C_total
    units_total = C_total if args.scaling == "strong" else C_total * world
    problem = Problem(arr)
    lib = _abi.lib()
    pk = peaks() if rank == 0 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing -----------------------------------------------------------------
    barrier()
    with ClockSampler(local) as clk:
        r = time_logdensity(problem, C, args.steps, args.warmup, args.radius, args.seed + 1 + rank,
                            use_graph=not args.no_graph, target_s=0, arr=arr if rank == 0 else None, pad_rows=args.pad_rows)
    barrier()
    ms = max_over_ranks(r["ms"])
    value = units_total * arr.num_matches * args.steps / (ms * 1e-3)
    last = r.pop("last")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last, suffix=f"_rank{rank}" if world > 1 else "")
    del last

    # ---- end to end (host buffers) ---------------------------------------------------------------------
    barrier()
    dt, h2d, d2h = time_e2e(problem, C, args.steps, args.warmup, args.radius, args.seed + 7 + rank)
    e2e_value = units_total * arr.num_matches * args.steps / max_over_ranks(dt)
    barrier()

    # ---- sub-records on all ranks -------------------------------------------------------------------------
    subs = []
    if not args.no_subrecords:
        problem_stats = problem.stats()
        for fn, a in ((sub_grid, (rank, world)), (sub_fit, (rank, world, args))):
            try:
                barrier()
                rec = fn(*a)
                if fn is sub_grid:
                    rec, flops = rec
                    if rank == 0:
                        rec["fp32_frac"] = flops / (rec["value"] * 1e-3) / 1e12 / pk["fp32_tflops"] / world
                subs.append(rec)
            except Exception as e:  # a sub-record must never lose the main line
                subs.append({"workload": fn.__name__, "error": repr(e)})
            torch.cuda.empty_cache()
    barrier()

    if rank == 0:
        st = problem.stats()
        t_launch = ms * 1e-3 / args.steps
        model = arr.model
        flops = FLOPS_PER_EVAL[model] * C * arr.num_matches
        ent_bytes = (16 if model == "extended" else 8) * st["entries1_padded"] + 8 * st["entries2_padded"]
        hbm_bytes = ent_bytes + 8 * problem.D * C + 8 * C  # static plan + theta in + grad out + lp, corr_coef
        smem_bytes = 8 * C * (st["entries1_padded"] + st["entries2_padded"])  # one float2 row read per chain-entry
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and world == 1:
            with open(tp) as f:
                traffic = (json.load(f).get(args.workload) or {}).get("traffic")  # dram read + write bytes of one launch (ncu --set full)
        roofline = {
            "bound": "fp32", "kernel": "bplx::logdensity_kernel",
            "achieved": flops / t_launch / 1e12, "peak": pk["fp32_tflops"], "unit": "TFLOP/s",
            "frac": flops / t_launch / 1e12 / pk["fp32_tflops"],
            "peak_source": "FFMA issue peak measured in this run (bench_kernels/fp32_peak.cu); "
                           "algorithmic flops/eval from SURVEY.md 8(d); per GPU (rank 0's shard and launch time)",
            "flops_per_eval": FLOPS_PER_EVAL[model], "traffic": traffic,
            "hbm": {"achieved": hbm_bytes / t_launch / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": hbm_bytes / t_launch / 1e9 / pk["hbm_gbs"], "algorithmic_bytes": hbm_bytes,
                    "peak_source": pk["hbm_source"]},
            "smem": {"achieved": smem_bytes / t_launch / 1e12, "peak": pk["smem_tbs"], "unit": "TB/s",
                     "frac": smem_bytes / t_launch / 1e12 / pk["smem_tbs"],
                     "peak_source": "LDS.64 peak measured in this run"},
        }
        groups = (C + 31) // 32
        # the CPU baseline is a reported number of the N=1 run only
        cpu = cpu_port(arr, C_total, args.cpu_chains, args.cpu_seconds, args.radius, args.seed + 1) if world == 1 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc + f", {C_total} chains " + (f"partitioned over {world} GPU(s)" if args.scaling == "strong" else "per GPU"),
                       "chains_total": units_total, "chains_per_gpu": C, "matches": arr.num_matches,
                       "teams": arr.num_teams, "params": problem.D, "theta": f"U(-{args.radius},{args.radius})",
                       "layout": f"chain-minor [D, C] resident in HBM, row pitch {r['ld']} floats",
                       "l2": f"inputs rotate through {r['nb']} buffer sets of {r['set_bytes'] / 1e6:.1f} MB each "
                             f"({r['nb'] * r['set_bytes'] / 1e6:.0f} MB > 126 MB L2)",
                       "timing": f"{'one replay of a CUDA graph of' if not args.no_graph else ''} {args.steps} launches, "
                                 "CUDA events on the launch stream, max over ranks",
                       "waves": {"chain_groups_per_gpu": groups, "sms": 148, "waves": groups / 148.0,
                                 "quantisation_efficiency": groups / (148.0 * math.ceil(groups / 148.0)),
                                 "launches_per_step": r["launches"] / max(args.steps, 1),
                                 "tail_split": ("the last partial wave (%d groups) runs as thread-block clusters in a second launch"
                                                % (groups % 148)) if r["launches"] > args.steps else "none"},
                       "plan": st},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.steps,
                    "api": "bplx_logdensity_fwdbwd_host (pinned numpy in/out, chain-major [C, D]; transposed on the device to "
                           "the native layout, copies and kernels pipelined in chunks)"},
            "gpu_launches": r["launches"],
            "finite": r["finite"],
            "parity_max_err": r["parity"],
            "roofline": roofline,
            "cpu_baseline": cpu,
            "sub_records": subs,
        }
        if world == 1 and not args.no_extras:
            try:
                line["extra_workloads"] = extras(args, pk)
            except Exception as e:  # extras must never lose the main line
                line["extra_workloads_error"] = repr(e)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
