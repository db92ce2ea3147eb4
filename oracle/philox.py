"""curand's Philox4_32_10 on the host -- the random numbers of ``csrc/nuts.cu``.

``stream(seed, subsequence, offset, n)`` returns the same 32-bit outputs as ``n`` calls of ``curand()`` after
``curand_init(seed, subsequence, offset, &state)``, vectorised over chains; ``uniform`` and ``box_muller`` restate
``_curand_uniform`` and ``_curand_box_muller`` (the uniform is the exact float32 value; the normals are float64, where the
device uses ``__sincosf`` and agrees to about 1e-6).  ``tests/test_nuts_reference.py`` checks all of it against curand's
own header code built for the host.
"""
from __future__ import annotations

import numpy as np

_M32 = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """Ten Philox rounds on the counter words ``ctr = (x, y, z, w)`` under ``key = (k0, k1)``.  The words are Python ints
    (one block, cheap) or uint64 numpy arrays of 32-bit values (one block per element); returns the 4 output words."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0 = 0xD2511F53 * c0  # 32 x 32 -> 64 bits: exact in uint64
        p1 = 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _M32, p1 & _M32, ((p0 >> 32) ^ c3 ^ k1) & _M32, p0 & _M32
        k0 = (k0 + 0x9E3779B9) & _M32
        k1 = (k1 + 0xBB67AE85) & _M32
    return c0, c1, c2, c3


def block(seed: int, subsequence: int, counter: int):
    """The four outputs at offsets ``4 counter .. 4 counter + 3`` of one sequence (Python ints)."""
    hi = subsequence + (counter >> 64)
    return philox4x32_10((counter & _M32, (counter >> 32) & _M32, hi & _M32, (hi >> 32) & _M32),
                         (seed & _M32, (seed >> 32) & _M32))


def stream(seed, subsequence, offset, n):
    """``[..., n]`` uint32: outputs ``offset .. offset + n - 1`` of the Philox sequence ``subsequence`` under key ``seed``
    (``curand_init`` + ``n`` x ``curand``).  The arguments broadcast against each other (one stream per chain)."""
    seed, sub, off = np.broadcast_arrays(*(np.asarray(a, dtype=np.uint64) for a in (seed, subsequence, offset)))
    key = (seed & _M32, seed >> 32)
    first = (off & 3).astype(np.int64)
    nblk = (int(first.max(initial=0)) + n + 3) // 4
    words = []
    for b in range(nblk):  # 128-bit counter offset / 4 + b + (subsequence << 64), carrying into the high half
        lo = (off >> 2) + np.uint64(b)
        hi = sub + (lo < np.uint64(b)).astype(np.uint64)
        words += philox4x32_10((lo & _M32, lo >> 32, hi & _M32, hi >> 32), key)
    words = np.stack(words, axis=-1).astype(np.uint32)  # [..., 4 nblk]
    return np.take_along_axis(words, first[..., None] + np.arange(n), axis=-1)


def uniform(x):
    """``_curand_uniform``: ``x * 2^-32 + 2^-33`` in float32, in (0, 1]."""
    return np.asarray(x, dtype=np.uint32).astype(np.float32) * np.float32(2.0 ** -32) + np.float32(2.0 ** -33)


def box_muller(x, y):
    """``_curand_box_muller(x, y)`` -> (n0, n1) in float64, from the float32 ``u`` and angle the device computes."""
    u = uniform(x)
    v = np.asarray(y, dtype=np.uint32).astype(np.float32) * np.float32(2.0 * np.pi * 2.0 ** -32) \
        + np.float32(2.0 * np.pi * 2.0 ** -33)
    s = np.sqrt(-2.0 * np.log(u.astype(np.float64)))
    v = v.astype(np.float64)
    return s * np.sin(v), s * np.cos(v)
