"""CPU: the pieces of the float64 reference NUTS (oracle/nuts.py) that the GPU comparison relies on -- curand's Philox
stream restated in numpy, numpyro's checkpoint indexing, and the reference sampler itself on a Gaussian target."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import nuts as on, philox


def _nvcc():
    return shutil.which(os.environ.get("NVCC", "nvcc"))


_CURAND_HOST = r"""
#define QUALIFIERS static __forceinline__ __host__ __device__
#include <curand_kernel.h>
#include <cstdio>
int main() {
  const unsigned long long seeds[3] = {0ull, 7ull, 0x123456789abcdefull};
  const unsigned long long subs[4] = {0ull, 5ull, 1000003ull, 0xfedcba9876ull};
  const unsigned long long offs[6] = {0ull, 1ull, 3ull, 64ull, 1029ull, 123456789011ull};
  for (auto s : seeds) for (auto q : subs) for (auto o : offs) {
    curandStatePhilox4_32_10_t st;
    curand_init(s, q, o, &st);
    printf("%llu %llu %llu", s, q, o);
    for (int i = 0; i < 7; i++) printf(" %u", curand(&st));
    curand_init(s, q, o, &st);
    printf(" %.9g", curand_uniform(&st));
    curand_init(s, q, o, &st);
    const float2 n = curand_normal2(&st);
    printf(" %.9g %.9g\n", n.x, n.y);
  }
}
"""


def test_philox_stream_matches_curand_host_code(tmp_path):
    """Raw outputs and uniforms bit for bit, normals to float32 rounding, at 72 (seed, subsequence, offset) triples:
    offsets that are not multiples of 4, a 64-bit seed, a subsequence above 2^32 and runs that cross Philox blocks."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found: curand's header code cannot be built for the host")
    src, exe = tmp_path / "curand_host.cu", tmp_path / "curand_host"
    src.write_text(_CURAND_HOST)
    r = subprocess.run([nvcc, "-O1", "-o", str(exe), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rows = [line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()]
    assert len(rows) == 72
    seed, sub, off = (np.array([int(x[i]) for x in rows], dtype=np.uint64) for i in range(3))
    raw = np.array([[int(v) for v in x[3:10]] for x in rows], dtype=np.uint32)
    got = philox.stream(seed, sub, off, 7)
    np.testing.assert_array_equal(got, raw)
    np.testing.assert_array_equal(philox.uniform(got[:, 0]), np.array([float(x[10]) for x in rows], dtype=np.float32))
    n0, n1 = philox.box_muller(got[:, 0], got[:, 1])
    want = np.array([[float(x[11]), float(x[12])] for x in rows])
    err = np.abs(np.stack([n0, n1], axis=1) - want) / np.maximum(1, np.abs(want))
    assert err.max() < 1e-5, err.max()
    # the scalar block the reference's per-chain stream uses
    for i in (0, 17, 71):
        if int(off[i]) % 4 == 0:
            assert list(philox.block(int(seed[i]), int(sub[i]), int(off[i]) // 4)) == list(raw[i, :4])


def test_leaf_idx_to_ckpt_idxs():
    """numpyro's checkpoint levels for leaves 0-63 of a subtree."""
    # hand-derived: (idx_min, idx_max) for leaves 0..15
    want = [(1, 0), (0, 0), (2, 1), (0, 1), (2, 1), (1, 1), (3, 2), (0, 2),
            (2, 1), (1, 1), (3, 2), (1, 2), (3, 2), (2, 2), (4, 3), (0, 3)]
    assert [on.leaf_idx_to_ckpt_idxs(n) for n in range(16)] == want
    # every leaf: an odd leaf n closes the subtrees of 2, 4, .., 2^k leaves ending at n (k = its trailing one bits); the
    # first leaf of each is even and stored its momentum at its own idx_max -- those are exactly levels idx_min..idx_max,
    # and no even leaf in between overwrote them
    for n in range(64):
        lo, hi = on.leaf_idx_to_ckpt_idxs(n)
        k = (n ^ (n + 1)).bit_length() - 1  # trailing one bits
        if n % 2 == 0:
            assert lo == hi + 1 and hi == bin(n).count("1")
            continue
        starts = [n + 1 - (1 << j) for j in range(1, k + 1)]
        levels = [on.leaf_idx_to_ckpt_idxs(s)[1] for s in starts]
        assert sorted(levels) == list(range(lo, hi + 1)), n
        for s, lv in zip(starts, levels):
            assert all(on.leaf_idx_to_ckpt_idxs(e)[1] != lv for e in range(s + 2, n + 1, 2)), (n, s)
    assert on.leaf_idx_to_ckpt_idxs(63) == (0, 5) and on.leaf_idx_to_ckpt_idxs(31) == (0, 4)


def test_reference_sampler_on_an_anisotropic_gaussian():
    """The reference with warm-up (dual averaging, one middle window) on independent normals of scales 0.3 .. 3: means
    within 5 Monte-Carlo standard errors, sds within 5 %, the adapted inverse mass is the variance, acceptance near the
    target and no divergences."""
    mu = np.array([0.0, 1.0, -2.0, 3.0, 0.5, -0.5])
    sd = np.array([1.0, 0.3, 3.0, 2.0, 0.5, 1.5])

    def potential(theta):
        zz = (theta - mu) / sd
        return -0.5 * (zz * zz).sum(1), -zz / sd

    C = 96
    rng = np.random.default_rng(0)
    cfg = on.Config(num_warmup=120, num_samples=50, seed=3, step_size=1.0)
    chains = on.sample(potential, mu + sd * rng.uniform(-2, 2, (C, 6)), cfg)
    x = np.stack([c.samples for c in chains])  # [C, N, D]
    assert all(c.transitions == 170 and np.isfinite(c.samples).all() for c in chains)
    # ESS from the lag-1..20 autocorrelation of the pooled chains (initial positive sequence)
    xc = x - x.mean(axis=(0, 1))
    var = (xc * xc).mean(axis=(0, 1))
    rho = [(xc[:, k:] * xc[:, :-k]).mean(axis=(0, 1)) / var for k in range(1, 20)]
    tau = 1 + 2 * np.sum(np.where(np.cumprod(np.array(rho) > 0, axis=0), rho, 0), axis=0)
    ess = x.shape[0] * x.shape[1] / tau
    assert ess.min() > 1500, ess
    z = np.abs(x.mean(axis=(0, 1)) - mu) / (sd / np.sqrt(ess))
    assert z.max() < 5, z
    np.testing.assert_allclose(x.reshape(-1, 6).std(axis=0), sd, rtol=0.05)
    n = 90  # the middle window of 120 warm-up steps
    assert on.adaptation_schedule(120) == [(0, 17), (18, 107), (108, 119)]
    imm = np.mean([c.inv_mass for c in chains], axis=0)
    np.testing.assert_allclose(imm, n / (n + 5) * sd ** 2 + 1e-3 * 5 / (n + 5), rtol=0.15)
    # chain by chain: Stan's regularised variance of the window's draws (unregularised would be 5.3 % off at n = 90)
    for c in chains:
        w = np.stack(c.positions[18:108])
        np.testing.assert_allclose(c.inv_mass, n / (n + 5) * w.var(axis=0, ddof=1) + 1e-3 * 5 / (n + 5), rtol=1e-10)
    acc = np.mean([c.accept for c in chains])
    assert 0.7 < acc < 0.95, acc
    assert sum(c.num_divergent for c in chains) == 0
