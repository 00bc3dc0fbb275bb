"""Prioritized experience replay (Schaul et al., 2016) restated without a tree, in float64 unless stated: what the device
sum/min tree of libsacx (csrc/sacx_per.cuh) must compute.

  priority          p = (delta + eps)^alpha,  delta = (|q1 - y| + |q2 - y|) / 2  (or a given |td|)
  sampling          row k of B draws u_k = (k + U_k) / B * sum(p) and takes the first slot whose inclusive prefix sum exceeds u_k;
                    u_k at or beyond the prefix sum's end (rounding) takes the last slot with p > 0
  weights           w = (p / p_min)^(-beta), p_min over the stored transitions (p > 0)
  beta schedule     beta(t) = min(1, beta0 + (1 - beta0) t / beta_steps); beta_steps = 0 keeps beta0
  write-back        rows in order, a slot named twice keeps the highest row's priority; p_max = max(p_max, every row's p)
"""
from __future__ import annotations

import numpy as np


def td_delta(q1, q2, y):
    q1, q2, y = (np.asarray(v, dtype=np.float64) for v in (q1, q2, y))
    return 0.5 * (np.abs(q1 - y) + np.abs(q2 - y))


def priority(delta, alpha, eps):
    return (np.abs(np.asarray(delta, dtype=np.float64)) + eps) ** alpha


def beta_at(t, beta0, beta_steps):
    if beta_steps == 0:
        return float(beta0)
    return min(1.0, beta0 + (1.0 - beta0) * t / beta_steps)


def strata_u(U, total):
    """u_k = (k + U_k) / B * total in float64."""
    U = np.asarray(U, dtype=np.float64)
    B = U.shape[0]
    return (np.arange(B) + U) / B * total


def strata_u_f32(U, total):
    """The same in the device's float32 arithmetic ((float)k + U) / (float)B * total: exact test vectors compare against this."""
    U = np.asarray(U, dtype=np.float32)
    B = np.float32(U.shape[0])
    return ((np.arange(U.shape[0], dtype=np.float32) + U) / B) * np.float32(total)


def sample(p, u):
    """Slots for draws u over priorities p (by slot, 0 = empty): first inclusive prefix sum > u, clamped to the last p > 0."""
    p = np.asarray(p, dtype=np.float64)
    c = np.cumsum(p)
    idx = np.searchsorted(c, np.asarray(u, dtype=np.float64), side="right")
    last = int(np.nonzero(p > 0)[0][-1])
    return np.minimum(idx, last)


def weights(p, p_sel, beta):
    p = np.asarray(p, dtype=np.float64)
    p_min = p[p > 0].min()
    return (np.asarray(p_sel, dtype=np.float64) / p_min) ** (-beta)


def write_back(leaves, slots, prios, p_max):
    """Sequential write-back (the highest row wins a duplicated slot); returns (new leaves, new p_max)."""
    out = np.array(leaves, dtype=np.float64, copy=True)
    for s, v in zip(np.asarray(slots), np.asarray(prios, dtype=np.float64)):
        out[int(s)] = v
    return out, max(float(p_max), float(np.max(prios))) if len(prios) else float(p_max)


def logical_to_slot(j, pushes, capacity):
    oldest = pushes % capacity if pushes > capacity else 0
    return (oldest + np.asarray(j)) % capacity
