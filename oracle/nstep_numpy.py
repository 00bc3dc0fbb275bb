"""n-step returns (``buffer.n_step``) restated in NumPy: what the gather of libsacx folds into every batch row
(csrc/sacx_math.cuh nstep_fold, called by op_gather and the row-parallel kernel's rp_nstep_fold).

For logical position j of a ring that holds L transitions (0 = oldest) and a discount gamma:
  m       the first i in 1..n with d[j+i-1] != 0, or i == n, or j+i-1 == L-1 (cut at a terminal, at n, at the newest record)
  R       r[j] + gamma r[j+1] + ... + gamma^(m-1) r[j+m-1]
  end     j + m - 1: the row's next state is s2[end]
  d_eff   1 if d[end] != 0, else 1 - gamma^(m-1)

``fold_f32`` is the device's float32 arithmetic, operation for operation (g_i = g_{i-1} * gamma, acc = acc + g_i r[j+i],
d_eff = 1 - g_{m-1}, each rounded to nearest; no fused multiply-add), so the kernels must match it bit for bit.
``fold_f64`` is the same quantity in float64, the semantic reference.
"""
from __future__ import annotations

import numpy as np


def window(d, j: int, n: int) -> int:
    """m, the length of the return window starting at logical position j (d: done column in logical order)."""
    L = len(d)
    for i in range(1, n + 1):
        k = j + i - 1
        if d[k] != 0 or i == n or k == L - 1:
            return i
    raise AssertionError("unreachable")


def fold_f32(r, d, j: int, n: int, gamma):
    """(R, d_eff, end) in the device's float32 order."""
    r = np.asarray(r, dtype=np.float32)
    g32 = np.float32(gamma)
    m = window(d, j, n)
    g, acc = np.float32(1.0), r[j]
    for i in range(1, m):
        g = np.float32(g * g32)
        acc = np.float32(acc + np.float32(g * r[j + i]))
    end = j + m - 1
    d_eff = np.float32(1.0) if d[end] != 0 else np.float32(np.float32(1.0) - g)
    return acc, d_eff, end


def fold_f64(r, d, j: int, n: int, gamma):
    """(R, d_eff, end) in float64 (gamma taken as the float32 value the engine stores)."""
    g = float(np.float32(gamma))
    m = window(d, j, n)
    R = sum(g ** i * float(r[j + i]) for i in range(m))
    end = j + m - 1
    return R, (1.0 if d[end] != 0 else 1.0 - g ** (m - 1)), end


def fold_batch_f32(r, d, idx, n: int, gamma):
    """Arrays (R [B], d_eff [B], end [B]) for the logical indices idx."""
    out = [fold_f32(r, d, int(j), n, gamma) for j in np.asarray(idx).reshape(-1)]
    return (np.array([o[0] for o in out], dtype=np.float32), np.array([o[1] for o in out], dtype=np.float32),
            np.array([o[2] for o in out], dtype=np.int64))


def target_f64(r, d, j: int, n: int, gamma, tq1, tq2, lp2, alpha) -> float:
    """The n-step soft target R + gamma^m (1 - d_end)(min(tq1, tq2) - alpha lp2) in float64, for the bootstrap terms
    (tq1, tq2, lp2) evaluated at s2[end]."""
    g = float(np.float32(gamma))
    m = window(d, j, n)
    R, _, end = fold_f64(r, d, j, n, gamma)
    return R + g ** m * (0.0 if d[end] != 0 else 1.0) * (min(float(tq1), float(tq2)) - float(alpha) * float(lp2))
