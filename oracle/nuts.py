"""Reference NUTS in float64 -- the checker of the GPU transition kernel (``csrc/nuts.cu``), written from numpyro's
algorithm (SURVEY.md Appendix C.5), not from the kernel: iterative subtree building with power-of-two checkpoints
(``_iterative_build_subtree``, ``_leaf_idx_to_ckpt_idxs``, ``_is_iterative_turning``), the uniform transition kernel inside
a subtree and the biased one at the top (``_combine_tree``), the generalised U-turn with a diagonal inverse mass,
divergence at dH > ``max_delta_energy`` (a NaN dH counts as +inf, a leaf whose log-density is not finite is rejected),
dual averaging (t0 = 10, kappa = 0.75, gamma = 0.05, mu = log 10 eps, ``exp(x_avg)`` after the last warm-up step) and
regularised Welford variances over Stan's windows (``bpl_next_b200.nuts.adaptation_schedule``).

Each chain is a generator that yields the position to evaluate and receives ``(lp, grad)``; ``sample`` evaluates the
positions of all live chains in one potential call per round.  One round is one ``bplx_nuts_step`` launch, so a chain
that consumes the kernel's random numbers follows the GPU chain draw for draw, up to rounding.

Random-number contract of the kernel (Philox4_32_10, key ``seed``, subsequence ``chain_offset + c``, ``oracle.philox``):

- per launch of a live chain, uniforms are drawn one after another from output offset ``rng_offset``, in this order:
  (1) the leaf-merge uniform, when the leaf is not the first of its subtree; (2) the trajectory-merge uniform, when a
  subtree completes; (3) the direction uniform (``u < 0.5``: right), when a new doubling starts;
- momentum refresh: ``r[d]`` is component ``d & 1`` of the Box-Muller pair at offset ``rng_offset + 64 + 4 (d >> 1)``,
  times ``rsqrt(inv_mass[d])``; a refresh counts ``64 + 2 D + 8`` draws;
- end of the launch: ``rng_offset += (draws + 7) & ~3`` (a launch without draws still advances it by 4);
- the first launch takes the log-density at the initial position, refreshes the momentum and picks a direction.

Every random or rounding-sensitive decision leaves a margin in the chain's trace: ``|u - p|`` for a uniform compared
with a probability, ``|v.s| / sum |v_i s_i|`` for a U-turn dot product, ``|dH - max_delta_energy| / max_delta_energy``
for a divergence test.  A float32 sampler may decide differently from this one only where a margin is small.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, List, Sequence

import numpy as np

from bpl_next_b200.nuts import adaptation_schedule

from . import philox

_TINY32 = float(np.finfo(np.float32).tiny)


def leaf_idx_to_ckpt_idxs(n: int):
    """numpyro ``_leaf_idx_to_ckpt_idxs``: the checkpoint levels ``idx_min .. idx_max`` leaf ``n`` of a subtree is tested
    against (``idx_max`` = set bits of ``n >> 1``, ``idx_min = idx_max - trailing ones of n + 1``); an even leaf is stored
    at ``idx_max``."""
    idx_max = bin(n >> 1).count("1")
    ones = 0
    while (n >> ones) & 1:
        ones += 1
    return idx_max - ones + 1, idx_max


@dataclass
class Config:
    num_warmup: int = 0
    num_samples: int = 10
    thin: int = 1
    max_tree_depth: int = 10
    target_accept: float = 0.8
    step_size: float = 1.0
    max_delta_energy: float = 1000.0
    seed: int = 42
    chain_offset: int = 0


@dataclass
class Chain:
    """What one reference chain produced, in the shapes of one chain of ``bpl_next_b200.nuts.NutsRun``."""
    samples: np.ndarray                  # [num_keep, D]
    lp: np.ndarray                       # [num_keep]
    accept: np.ndarray                   # [num_keep]
    inv_mass: np.ndarray                 # [D]
    step_size: float = 0.0
    num_divergent: int = 0
    num_leapfrog: int = 0
    transitions: int = 0
    # decisions: (transition, kind, margin, detail) for every rounding-sensitive decision
    decisions: List[tuple] = field(default_factory=list)
    leapfrogs: List[int] = field(default_factory=list)  # per transition
    positions: List[np.ndarray] = field(default_factory=list)  # the draw of every transition, warm-up included
    # coverage: most trailing one bits of a tested leaf index, depth-limit hits, subtrees that turned before their last
    # leaf, top-level merges rejected by their uniform, divergent leaves, leaves with a non-finite log-density
    max_trailing_ones: int = 0
    depth_limit_hits: int = 0
    early_subtree_turns: int = 0
    rejected_merges: int = 0
    divergences: int = 0
    nonfinite_leaves: int = 0

    def min_margin(self, first: int, last: int) -> float:
        """Smallest decision margin at transitions ``first .. last``."""
        return min((m for t, _, m, _ in self.decisions if first <= t <= last), default=math.inf)

    def history(self, t: int) -> str:
        return "; ".join(f"{k} margin {m:.2e} ({s})" for tt, k, m, s in self.decisions if tt == t) or "no decisions"


class _Rng:
    """The kernel's per-chain Philox stream as a chain consumes it, launch by launch."""

    def __init__(self, seed: int, sub: int):
        self.seed, self.sub = seed, sub
        self.offset = 0  # at the start of the current launch; always a multiple of 4
        self.draws = self.nu = 0
        self.words = None

    def uniform(self) -> float:
        if self.words is None:
            self.words = philox.block(self.seed, self.sub, self.offset >> 2)
        assert self.nu < 4
        u = float(philox.uniform(self.words[self.nu]))
        self.nu += 1
        self.draws += 1
        return u

    def normals(self, D: int) -> np.ndarray:
        ctr = np.uint64((self.offset + 64) >> 2) + np.arange((D + 1) // 2, dtype=np.uint64)
        k = (self.seed & 0xFFFFFFFF, self.seed >> 32)
        w0, w1, _, _ = philox.philox4x32_10((ctr & 0xFFFFFFFF, ctr >> 32, np.uint64(self.sub & 0xFFFFFFFF),
                                             np.uint64(self.sub >> 32)), tuple(np.uint64(x) for x in k))
        n0, n1 = philox.box_muller(w0, w1)
        self.draws += 64 + 2 * D + 8
        return np.stack([n0, n1], axis=1).reshape(-1)[:D]

    def end_launch(self):
        self.offset += (self.draws + 7) & ~3
        self.draws = self.nu = 0
        self.words = None


def _exp(x: float) -> float:
    return math.exp(x) if x < 709.0 else math.inf


def _sigmoid(x: float) -> float:
    if x >= 0:
        return 1.0 / (1.0 + math.exp(-x))
    e = math.exp(x) if x == x else math.nan
    return e / (1.0 + e)


def _logaddexp(a: float, b: float) -> float:
    m = max(a, b)
    if m == -math.inf:
        return m
    return m + math.log1p(math.exp(-abs(a - b)))


def _dot_margin(v, s) -> float:
    den = float(np.abs(v * s).sum())
    return abs(float(v @ s)) / den if den > 0 else 0.0


def _turning(im, r_left, r_right, r_sum):
    """numpyro ``_is_turning`` (diagonal inverse mass) -> (turning, margin of the decision)."""
    s = r_sum - 0.5 * (r_left + r_right)
    vl, vr = im * r_left, im * r_right
    dl, dr = float(vl @ s), float(vr @ s)
    ml, mr = _dot_margin(vl, s), _dot_margin(vr, s)
    if dl <= 0 or dr <= 0:  # decided by the clearest of the products that turned
        return True, max(m for d, m in ((dl, ml), (dr, mr)) if d <= 0)
    return False, min(ml, mr)


def _chain(theta0: np.ndarray, cfg: Config, sub: int, out: Chain):
    """One chain; yields positions, receives (lp, grad)."""
    D = theta0.size
    rng = _Rng(cfg.seed, sub)
    im = np.ones(D)
    lp, g = yield theta0
    z, pe, zg = np.array(theta0, dtype=np.float64), -float(lp), np.asarray(g, dtype=np.float64)
    step = cfg.step_size
    da_mu, da_x, da_xavg, da_gavg, da_t = math.log(10 * step), 0.0, 0.0, 0.0, 0
    wf_mean, wf_m2, wf_n = np.zeros(D), np.zeros(D), 0
    sched, window = adaptation_schedule(cfg.num_warmup), 0
    mde = cfg.max_delta_energy
    for t in range(cfg.num_warmup + cfg.num_samples):
        def note(kind, margin, detail):
            out.decisions.append((t, kind, margin, detail))

        r = rng.normals(D) / np.sqrt(im)
        energy = pe + 0.5 * float((im * r) @ r)
        zL, rL, gL = z, r, zg
        zR, rR, gR = z, r, zg
        r_sum = r.copy()
        depth, weight, turning, diverging, sum_acc, nprop = 0, 0.0, False, False, 0.0, 0
        while True:  # doublings
            right = rng.uniform() < 0.5
            eps = step if right else -step
            ck, cks = np.zeros((cfg.max_tree_depth, D)), np.zeros((cfg.max_tree_depth, D))
            n_leaves = 1 << depth
            s_w, s_acc, s_sum, s_turn, s_div = 0.0, 0.0, None, False, False
            for n in range(n_leaves):  # _iterative_build_subtree
                z0, r0, g0 = (zR, rR, gR) if right else (zL, rL, gL)
                rh = r0 + 0.5 * eps * g0
                th = z0 + eps * im * rh
                rng.end_launch()
                lp1, g1 = yield th
                lp1, g1 = float(lp1), np.asarray(g1, dtype=np.float64)
                r1 = rh + 0.5 * eps * g1
                if right:
                    zR, rR, gR = th, r1, g1
                else:
                    zL, rL, gL = th, r1, g1
                pe1 = -lp1
                delta = pe1 + 0.5 * float((im * r1) @ r1) - energy
                if not math.isfinite(lp1) or delta != delta:
                    out.nonfinite_leaves += 1
                    delta = math.inf
                w = -delta
                acc = min(1.0, _exp(-delta))
                if n == 0:
                    take, s_w = True, w
                else:  # uniform transition kernel inside the subtree
                    p = _sigmoid(w - s_w)
                    u = rng.uniform()
                    take = u < p
                    note("leaf merge", abs(u - p), f"leaf {n} u={u:.6f} p={p:.6f}")
                    s_w = _logaddexp(s_w, w)
                if take:
                    s_prop = (th, pe1, g1)
                s_div = delta > mde
                note("divergence", abs(delta - mde) / mde, f"leaf {n} dH={delta:.6g}")
                out.divergences += s_div
                s_acc += acc
                s_sum = r1.copy() if n == 0 else s_sum + r1
                idx_min, idx_max = leaf_idx_to_ckpt_idxs(n)
                if n % 2 == 0:
                    ck[idx_max], cks[idx_max] = r1, s_sum
                else:
                    out.max_trailing_ones = max(out.max_trailing_ones, idx_max - idx_min + 1)
                for i in range(idx_max, idx_min - 1, -1):  # _is_iterative_turning: stop at the first turn
                    s_turn, m = _turning(im, ck[i], r1, s_sum - cks[i] + ck[i])
                    note("subtree U-turn", m, f"leaf {n} level {i} turning={s_turn}")
                    if s_turn:
                        break
                if s_turn or s_div:
                    out.early_subtree_turns += s_turn and n + 1 < n_leaves
                    break
            built = n + 1
            # _combine_tree with the biased transition kernel
            p = 0.0 if (s_turn or s_div) else min(1.0, _exp(s_w - weight))
            u = rng.uniform()
            move = u < p
            if p > 0:
                note("trajectory merge", abs(u - p), f"depth {depth} u={u:.6f} p={p:.6f}")
                out.rejected_merges += not move
            r_sum = r_sum + s_sum
            if move:
                z, pe, zg = s_prop
            whole, m = _turning(im, rL, rR, r_sum)
            note("trajectory U-turn", m, f"depth {depth} turning={whole}")
            turning = s_turn or whole
            depth += 1
            weight = _logaddexp(weight, s_w)
            diverging = s_div
            sum_acc += s_acc
            nprop += built
            if depth >= cfg.max_tree_depth or turning or diverging:
                out.depth_limit_hits += not (turning or diverging)
                break
        accept = sum_acc / nprop
        out.num_leapfrog += nprop
        out.leapfrogs.append(nprop)
        out.positions.append(z)
        if t >= cfg.num_warmup:
            out.num_divergent += diverging
            k = t - cfg.num_warmup
            if k % cfg.thin == 0 and k // cfg.thin < out.samples.shape[0]:
                out.samples[k // cfg.thin], out.lp[k // cfg.thin], out.accept[k // cfg.thin] = z, -pe, accept
        else:  # numpyro warmup_adapter: dual averaging, then Welford in the middle windows
            da_t += 1
            tt = float(da_t)
            da_gavg = (1 - 1 / (tt + 10)) * da_gavg + (cfg.target_accept - accept) / (tt + 10)
            da_x = da_mu - math.sqrt(tt) / 0.05 * da_gavg
            wt = tt ** -0.75
            da_xavg = (1 - wt) * da_xavg + wt * da_x
            step = max(_exp(da_xavg if t == cfg.num_warmup - 1 else da_x), _TINY32)
            at_end = t == sched[window][1]
            if 0 < window < len(sched) - 1:
                wf_n += 1
                pre = z - wf_mean
                wf_mean = wf_mean + pre / wf_n
                wf_m2 = wf_m2 + pre * (z - wf_mean)
                if at_end:
                    nn = float(wf_n)
                    im = (nn / (nn + 5)) * (wf_m2 / (nn - 1)) + 1e-3 * (5 / (nn + 5))
                    wf_mean, wf_m2, wf_n = np.zeros(D), np.zeros(D), 0
                    da_mu, da_x, da_xavg, da_gavg, da_t = math.log(10 * step), 0.0, 0.0, 0.0, 0
            window += at_end
        out.transitions = t + 1
    out.step_size, out.inv_mass = step, im


def sample(potential: Callable[[np.ndarray], tuple], theta0: np.ndarray, cfg: Config,
           chains: Sequence[int] = None) -> List[Chain]:
    """Run the reference for the chains ``chains`` (global indices ``c``: subsequence ``cfg.chain_offset + c``) from
    ``theta0 [len(chains), D]``.  ``potential(theta [n, D]) -> (lp [n], grad [n, D])`` in float64, one call per round."""
    theta0 = np.asarray(theta0, dtype=np.float64)
    n, D = theta0.shape
    chains = list(range(n)) if chains is None else list(chains)
    num_keep = (cfg.num_samples + cfg.thin - 1) // cfg.thin
    outs = [Chain(samples=np.full((num_keep, D), np.nan), lp=np.full(num_keep, np.nan), accept=np.full(num_keep, np.nan),
                  inv_mass=np.ones(D)) for _ in range(n)]
    gens = [_chain(theta0[i], cfg, cfg.chain_offset + c, outs[i]) for i, c in enumerate(chains)]
    pos = {i: next(g) for i, g in enumerate(gens)}
    while pos:
        live = sorted(pos)
        lp, grad = potential(np.stack([pos[i] for i in live]))
        for j, i in enumerate(live):
            try:
                pos[i] = gens[i].send((lp[j], grad[j]))
            except StopIteration:
                del pos[i]
    return outs
