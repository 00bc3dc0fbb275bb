"""CPU tests of the float32 restatement of the prioritized-replay tree (oracle/per_numpy.py tree_f32 / walk_f32 / beta_f32) and
of its Philox stream (oracle/device_rng.py per_uniform), which test_gpu_per_oracle.py compares the device with bit for bit.

Rounding bound of a draw. The float32 walk and the float64 `sample()` agree except where a draw lies within rounding of a
prefix boundary. Every value involved is a sum of non-negative terms, so each float32 operation errs by at most
u = 2^-24 of `total`:
- the draw u_k = ((k + U) / B) * total: 3 roundings, and `total` itself, a butterfly of 5 adds per level: 5 depth;
- per level of the walk: the scan (5 adds), sc_f - v_f (1), u - before (1), and the children's own butterfly sums (5).
That is at most (3 + 17 depth) u total (first order); `walk_bound` returns it, and the draws within it of a boundary are
flagged, not compared.
"""
import numpy as np
import pytest

from oracle import device_rng as R
from oracle import per_numpy as P

F32 = np.float32
U24 = 2.0 ** -24


def walk_bound(levels, extra_rel=0.0):
    """(3 + 17 depth) 2^-24 total, plus extra_rel total (relative error of the leaves themselves, if any)."""
    depth = len(levels) - 1
    return ((3 + 17 * depth) * U24 + extra_rel) * float(levels[-1][0][0])


def check_walk(leaves, U, extra_rel=0.0):
    """walk_f32 against float64 sample(): equal off the flagged draws, a neighbour of the boundary on them; never p = 0.
    Returns the number of flagged draws."""
    lv = P.tree_f32(leaves)
    got = P.walk_f32(lv, U)
    p = leaves.astype(np.float64)
    u = P.strata_u(U, p.sum())
    tol = walk_bound(lv, extra_rel)
    flag = P.boundary_rows(p, u, tol)
    want = P.sample(p, u)
    assert np.array_equal(got[~flag], want[~flag])
    lo, hi = P.sample(p, np.maximum(u - tol, 0)), P.sample(p, u + tol)
    assert np.all((got >= lo) & (got <= hi))
    assert np.all(p[got] > 0)
    return int(flag.sum())


def profile(rng, n, zeros=0.1):
    """(delta + eps)^alpha of deltas over four decades, with zeros (empty slots) mixed in, as float32."""
    delta = 10.0 ** rng.uniform(-3, 1, n)
    p = ((delta + 1e-6) ** 0.6).astype(F32)
    p[rng.random(n) < zeros] = 0
    p[rng.integers(0, n)] = F32(1.5)
    return p


@pytest.mark.parametrize("cap,fill", [(1, 1), (31, 31), (32, 20), (33, 33), (1025, 1025), (5000, 3100), (1 << 17, 1 << 17)])
def test_walk_f32_matches_float64_sampling_off_the_boundaries(cap, fill):
    rng = np.random.default_rng(cap)
    leaves = np.zeros(cap, F32)
    leaves[:fill] = profile(rng, fill)
    flagged = 0
    for B in (1, 7, 256, 4096):
        U = rng.random(B).astype(F32)
        U[0], U[-1] = 0.0, F32(1 - U24)
        flagged += check_walk(leaves, U)
    print(f"cap {cap}: {flagged} of {1 + 7 + 256 + 4096} draws within {walk_bound(P.tree_f32(leaves)) / leaves.sum():.2e} "
          f"total of a boundary")


def test_tree_f32_of_integer_leaves_is_exact():
    """Integer leaves below 2^24 in total: every node's sum is exact, the min is the smallest nonzero child."""
    rng = np.random.default_rng(3)
    for cap in (1, 32, 33, 1025, 40000):
        leaves = rng.integers(0, 9, cap).astype(F32)
        leaves[0] = 1
        lv = P.tree_f32(leaves)
        exact = leaves.astype(np.float64)
        ex_min = np.where(exact > 0, exact, np.inf)
        for l in range(1, len(lv)):
            n = len(lv[l][0])
            pad = n * 32 - len(exact)
            exact = np.concatenate([exact, np.zeros(pad)]).reshape(n, 32).sum(axis=1)
            ex_min = np.concatenate([ex_min, np.full(pad, np.inf)]).reshape(n, 32).min(axis=1)
            assert np.array_equal(lv[l][0], exact) and np.array_equal(lv[l][1], ex_min), (cap, l)
        assert len(lv[-1][0]) == 1 and len(lv) - 1 == max(1, int(np.ceil(np.log(cap) / np.log(32) - 1e-12)))


def test_fallback_takes_the_last_nonzero_child():
    """A draw at or past the scan's own last prefix sum (the root's butterfly total can round above it) takes the last child
    with p > 0, not lane 31 and not an empty slot."""
    rng = np.random.default_rng(11)
    for _ in range(20000):
        leaves = np.zeros(32, F32)
        leaves[:20] = rng.uniform(0.1, 3, 20).astype(F32)
        sc = leaves.copy()
        for off in (1, 2, 4, 8, 16):
            t = sc.copy(); t[off:] = sc[off:] + sc[:-off]; sc = t
        lv = P.tree_f32(leaves)
        if sc[-1] < lv[-1][0][0]:
            break
    else:
        pytest.fail("no leaves whose scan ends below the butterfly total")
    total = lv[-1][0][0]
    U = np.array([1 - U24], F32)
    assert (U * total).astype(F32)[0] >= sc[-1]               # the draw is past every scanned prefix sum
    assert P.walk_f32(lv, U)[0] == 19


def start_trap():
    """(leaves, U): root children 1 and 1 + 3 2^-23, whose scanned sum rounds to 2 + 2^-21, so sc_1 - v_1 = 1 + 2^-23 > sc_0.
    The draw u = 1 (= sc_0, not past it) leaves u = -2^-23 inside child 1, whose first slot (32) is empty."""
    leaves = np.zeros(64, F32)
    leaves[0], leaves[33] = 1, F32(1 + 3 * 2.0 ** -23)
    return leaves, np.array([8388606 * U24], F32)


def end_trap():
    """(leaves, U): a partly filled 32-slot ring whose scan over the empty slot 20 rounds above its sum over slots 0..19, and
    a last-stratum draw between the two."""
    rng = np.random.default_rng(5)
    for _ in range(100000):
        leaves = np.zeros(32, F32)
        leaves[:20] = rng.uniform(0.1, 3, 20).astype(F32)
        sc = leaves.copy()
        for off in (1, 2, 4, 8, 16):
            t = sc.copy(); t[off:] = sc[off:] + sc[:-off]; sc = t
        total = P.tree_f32(leaves)[-1][0][0]
        for m in range(1, 64):
            U = np.array([1 - m * U24], F32)
            u = (U * total)[0]
            if sc[19] <= u < sc[20]:
                return leaves, U
    raise AssertionError("no such leaves")


def test_rounding_never_takes_an_empty_slot():
    """At both traps the first child with sc > u is empty (p = 0): the walk takes the first child with p > 0 and sc > u
    instead, slot 33 at the start trap and the last stored slot 19 at the end trap."""
    leaves, U = start_trap()
    lv = P.tree_f32(leaves)
    assert ((U / F32(1)) * lv[-1][0][0])[0] == F32(1)
    assert P.walk_f32(lv, U)[0] == 33
    leaves, U = end_trap()
    assert P.walk_f32(P.tree_f32(leaves), U)[0] == 19


def test_beta_f32_follows_the_schedule():
    for t, steps, want in ((0, 0, F32(0.4)), (10 ** 9, 0, F32(0.4)), (0, 100, F32(0.4)), (99, 100, F32(0.4 + 0.6 * 99 / 100)),
                           (100, 100, F32(1)), (101, 100, F32(1))):
        assert P.beta_f32(t, 0.4, steps) == want, (t, steps)
    # beta0 enters as the float32 the tree was created with, widened to double
    assert P.beta_f32(1, 0.3, 3) == F32(float(F32(0.3)) + (1 - float(F32(0.3))) / 3)


def test_per_uniform_is_24_bit_uniform_and_its_own_stream():
    seed, counter, agent = 0x0123456789ABCDEF, 2 ** 32 + 17, 5
    u = R.per_uniforms(seed, counter, 1 << 16, agent)
    assert u.dtype == np.float32 and u.min() >= 0 and u.max() < 1
    assert np.array_equal(u * F32(2 ** 24), np.floor(u * F32(2 ** 24)))          # 24-bit values
    n = len(u)
    assert abs(u.mean() - 0.5) < 5 * np.sqrt(1 / 12 / n)
    assert abs(u.var() - 1 / 12) < 5 * np.sqrt(1 / 180 / n)
    for k in (0, 1, 31, 65535):
        assert u[k] == R.per_uniform(seed, counter, k, agent)
    # keyed by every argument
    assert not np.array_equal(u[:64], R.per_uniforms(seed, counter + 1, 64, agent))
    assert not np.array_equal(u[:64], R.per_uniforms(seed, counter, 64, agent + 1))
    assert not np.array_equal(u[:64], R.per_uniforms(seed + 1, counter, 64, agent))
    # not the policy-noise stream of the same (seed, counter, row)
    for k in range(8):
        u1, u2 = R.philox_uniforms(seed, counter, 1, k, 0, agent)
        assert u[k] not in (u1, u2)
