"""Oracle (test infrastructure only): NumPy restatement of the device RNG streams of the throughput mode.

``csrc/sacx_math.cuh`` draws, inside the update kernels, the batch indices with a keyed Feistel bijection on [0, n) and the
policy noise with Philox4x32-10 followed by Box-Muller. This module restates both with Python integers, so the index
stream is reproduced bit for bit; the normal's two uniforms go through the same float32 conversions as the device code and
Box-Muller is then evaluated in float64 (the device's float32 ``logf`` / ``cospif`` differ from it by a few ulps).
"""
from __future__ import annotations

import math

import numpy as np

_M32 = 0xFFFFFFFF
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4x32_10(ctr, key):
    """Philox4x32 with 10 rounds (Salmon et al., SC'11): ctr 4 words, key 2 words -> 4 words."""
    c0, c1, c2, c3 = (int(x) & _M32 for x in ctr)
    k0, k1 = (int(x) & _M32 for x in key)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & _M32, (p0 >> 32) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + _W0) & _M32, (k1 + _W1) & _M32
    return [c0, c1, c2, c3]


def philox_uniforms(seed, update, which, row, j, agent):
    """(u1, u2) as float32, exactly as ``philox_normal`` forms them: u1 in (0, 1], u2 in [0, 1)."""
    seed, update = int(seed), int(update)
    o = philox4x32_10((update & _M32, (update >> 32) & _M32, row, ((which << 24) | j) & _M32),
                      ((seed & _M32) ^ ((agent * 0x9E3779B9) & _M32), ((seed >> 32) & _M32) ^ 0x5AC5AC5A))
    f = np.float32
    u1 = (f(o[0]) + f(1.0)) * f(2.3283064365386963e-10)
    u2 = f(o[1]) * f(2.3283064365386963e-10)
    u1 = min(max(u1, f(1e-30)), f(1.0))
    return f(u1), f(u2)


def per_uniform(seed, counter, k, agent):
    """U[0, 1) of row k of prioritized-replay draw `counter` (``per_uniform`` in csrc/sacx_per.cuh): the Philox stream tagged
    0x7E in counter word 3, top 24 bits of word 0 times 2^-24 (exact in float32)."""
    seed, counter = int(seed), int(counter)
    o = philox4x32_10((counter & _M32, (counter >> 32) & _M32, k, 0x7E000000),
                      ((seed & _M32) ^ ((agent * 0x9E3779B9) & _M32), ((seed >> 32) & _M32) ^ 0x5AC5AC5A))
    return np.float32(o[0] >> 8) * np.float32(5.9604644775390625e-8)


def per_uniforms(seed, counter, B, agent):
    """per_uniform(seed, counter, k, agent) for k = 0 .. B-1 as a float32 array: the same rounds on uint64 lanes."""
    seed, counter = int(seed), int(counter)
    m32 = np.uint64(_M32)
    u = lambda x: np.uint64(int(x) & _M32)
    c0 = np.full(B, u(counter), np.uint64)
    c1 = np.full(B, u(counter >> 32), np.uint64)
    c2 = np.arange(B, dtype=np.uint64)
    c3 = np.full(B, np.uint64(0x7E000000), np.uint64)
    k0, k1 = (seed & _M32) ^ ((agent * 0x9E3779B9) & _M32), ((seed >> 32) & _M32) ^ 0x5AC5AC5A
    for _ in range(10):
        p0, p1 = np.uint64(_M0) * c0, np.uint64(_M1) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ u(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ u(k1), p0 & m32
        k0, k1 = (k0 + _W0) & _M32, (k1 + _W1) & _M32
    return (c0 >> np.uint64(8)).astype(np.float32) * np.float32(5.9604644775390625e-8)


def philox_normal(seed, update, which, row, j, agent):
    """N(0, 1) draw of element (update, which, row, j): Box-Muller in float64 on the device's float32 uniforms."""
    u1, u2 = philox_uniforms(seed, update, which, row, j, agent)
    return math.sqrt(-2.0 * math.log(float(u1))) * math.cos(2.0 * math.pi * float(u2))


def _mix32(x):
    x ^= x >> 16
    x = (x * 0x85EBCA6B) & _M32
    x ^= x >> 13
    x = (x * 0xC2B2AE35) & _M32
    x ^= x >> 16
    return x


def feistel_key(seed, counter, agent):
    """Round keys of one update: one Philox block per (update counter, agent, seed)."""
    seed, counter = int(seed), int(counter)
    return philox4x32_10((counter & _M32, (counter >> 32) & _M32, 0x1D8E4E27, agent), (seed & _M32, (seed >> 32) & _M32))


def feistel_apply(i, n, key):
    """Position i in [0, n) -> a distinct element of [0, n): six-round balanced Feistel network with cycle walking."""
    i, n = int(i), int(n)
    if n <= 1:
        return 0
    bits = (n - 1).bit_length()
    half = max((bits + 1) >> 1, 1)
    mask = _M32 if half >= 32 else (1 << half) - 1
    x = i
    while True:
        L, R = (x >> half) & mask, x & mask
        for r in range(6):
            f = _mix32((R ^ key[r & 3] ^ ((0x9E3779B9 * (r + 1)) & _M32)) & _M32) & mask
            L, R = R, L ^ f
        x = (L << half) | R
        if x < n:
            return x


def feistel_index(i, n, seed, counter, agent):
    return feistel_apply(i, n, feistel_key(seed, counter, agent))


def feistel_indices(count, n, seed, counter, agent):
    """feistel_index(i, ...) for i = 0 .. count-1 as an int64 array: the same network on uint64 lanes (whole domains of a
    million positions in well under a second)."""
    n = int(n)
    if n <= 1:
        return np.zeros(count, np.int64)
    key = [np.uint64(k) for k in feistel_key(seed, counter, agent)]
    bits = (n - 1).bit_length()
    half = max((bits + 1) >> 1, 1)
    mask = np.uint64(_M32 if half >= 32 else (1 << half) - 1)
    m32, sh = np.uint64(_M32), np.uint64(half)

    def mix(x):
        x ^= x >> np.uint64(16)
        x = (x * np.uint64(0x85EBCA6B)) & m32
        x ^= x >> np.uint64(13)
        x = (x * np.uint64(0xC2B2AE35)) & m32
        return x ^ (x >> np.uint64(16))

    out = np.arange(count, dtype=np.uint64)
    todo = np.ones(count, bool)
    while todo.any():
        x = out[todo]
        L, R = (x >> sh) & mask, x & mask
        for r in range(6):
            f = mix(R ^ key[r & 3] ^ np.uint64((0x9E3779B9 * (r + 1)) & _M32)) & mask
            L, R = R, L ^ f
        out[todo] = (L << sh) | R
        todo = out >= np.uint64(n)
    return out.astype(np.int64)
