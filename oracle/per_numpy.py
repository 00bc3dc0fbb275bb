"""Prioritized experience replay (Schaul et al., 2016) restated without a tree, in float64 unless stated: what the device
sum/min tree of libsacx (csrc/sacx_per.cuh) must compute.

  priority          p = (delta + eps)^alpha,  delta = (|q1 - y| + |q2 - y|) / 2  (or a given |td|)
  sampling          row k of B draws u_k = (k + U_k) / B * sum(p) and takes the first slot whose inclusive prefix sum exceeds u_k;
                    u_k at or beyond the prefix sum's end (rounding) takes the last slot with p > 0; a slot with p = 0 is
                    never taken
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


# ---------------------------------------------------------------------------------------------- float32 restatement
# The device tree and walk in the device's own float32 arithmetic: adds, one correctly rounded divide and one multiply (the
# library is built without fast-math), so the slot a draw takes is restated bit for bit. Only the weights' powf is not.
FANOUT = 32
F32 = np.float32


def tree_f32(leaves):
    """[(sum, min) of every level]: level 0 is (leaves, leaves with 0 -> +inf); level l >= 1 reduces groups of 32 nodes of
    level l - 1 by the xor butterfly of per_node (offsets 16, 8, 4, 2, 1; lane 0's value), zero-padded (min: +inf) past the
    last node, up to the single root node."""
    leaves = np.asarray(leaves, dtype=F32)
    levels = [(leaves, np.where(leaves > 0, leaves, F32(np.inf)).astype(F32))]
    lane = np.arange(FANOUT)
    while True:
        s, m = levels[-1]
        n = (len(s) + FANOUT - 1) // FANOUT
        ps = np.zeros(n * FANOUT, F32); ps[:len(s)] = s
        pm = np.full(n * FANOUT, np.inf, F32); pm[:len(m)] = m
        ps, pm = ps.reshape(n, FANOUT), pm.reshape(n, FANOUT)
        for off in (16, 8, 4, 2, 1):
            ps = ps + ps[:, lane ^ off]
            pm = np.minimum(pm, pm[:, lane ^ off])
        levels.append((ps[:, 0].copy(), pm[:, 0].copy()))
        if n == 1:
            return levels


def walk_f32(levels, U):
    """Slots the device walk takes for draws U (row k of B = len(U)): u = ((f32)k + U) / (f32)B * total; per level the
    inclusive Hillis-Steele scan of the 32 children (sc += shfl_up(sc, off), off = 1 .. 16), the first child with v > 0 and
    sc > u, u <- u - (sc_f - v_f); no such child (u within rounding of the node's sum): the last child with v > 0, u <- v_f.
    An empty child's scanned sum can round above its left neighbour's, and u - (sc_f - v_f) can round below 0: without the
    v > 0 condition either would take an empty slot."""
    U = np.asarray(U, dtype=F32)
    B = len(U)
    total = levels[-1][0][0]
    u = ((np.arange(B, dtype=F32) + U) / F32(B)) * total
    node = np.zeros(B, np.int64)
    lane = np.arange(FANOUT)
    for l in range(len(levels) - 1, 0, -1):
        child = levels[l - 1][0]
        c = node[:, None] * FANOUT + lane[None, :]
        v = np.where(c < len(child), child[np.minimum(c, len(child) - 1)], F32(0)).astype(F32)
        sc = v.copy()
        for off in (1, 2, 4, 8, 16):
            t = sc.copy()
            t[:, off:] = sc[:, off:] + sc[:, :-off]
            sc = t
        nz = v > 0
        hitm = (sc > u[:, None]) & nz
        hit = hitm.any(axis=1)
        last_nz = np.where(nz.any(axis=1), FANOUT - 1 - np.argmax(nz[:, ::-1], axis=1), 0)
        f = np.where(hit, np.argmax(hitm, axis=1), last_nz)
        r = np.arange(B)
        before, vf = (sc[r, f] - v[r, f]).astype(F32), v[r, f]
        u = np.where(hit, (u - before).astype(F32), vf).astype(F32)
        node = node * FANOUT + f
    return node


def beta_f32(t, beta0, beta_steps):
    """The device's beta(t): fmin(1, beta0 + (1 - beta0) t / beta_steps) in double, then a float32 cast (beta0 as the
    double the tree holds: sacx_per_create takes it as a float)."""
    beta0 = float(F32(beta0))
    if beta_steps <= 0:
        return F32(beta0)
    return F32(min(1.0, beta0 + (1.0 - beta0) * float(t) / float(beta_steps)))


def boundary_rows(p, u, tol):
    """Draws u within tol of an inclusive prefix sum of p (float64): a float32 walk may take either neighbour there."""
    c = np.cumsum(np.asarray(p, dtype=np.float64))
    c = c[np.concatenate([[True], np.diff(c) > 0])]
    u = np.asarray(u, dtype=np.float64)
    i = np.clip(np.searchsorted(c, u), 1, len(c) - 1)
    return np.minimum(np.abs(u - c[i - 1]), np.abs(u - c[i])) <= tol
