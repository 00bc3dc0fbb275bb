"""n-step returns without a device: ``buffer.n_step`` validation, the C config field, and the float64 / float32 restatements of
the fold (oracle/nstep_numpy.py) on hand-computed cases."""
import copy
import ctypes as C

import numpy as np
import pytest

from oracle import nstep_numpy as N


def _cfg(n_step="absent"):
    from gpu_helpers import base_config
    cfg = base_config(hidden=(32, 32), batch=16)
    if n_step != "absent":
        cfg["buffer"]["n_step"] = n_step
    return cfg


@pytest.mark.parametrize("value,want", [("absent", 1), (None, 1), (1, 1), (3, 3), (16, 16), (np.int64(5), 5)])
def test_yaml_accepts(value, want):
    from sac import _engine as E
    cfg = _cfg(value)
    assert E.n_step_config(cfg) == want
    assert E.make_config(4, 2, cfg).n_step == want


@pytest.mark.parametrize("value", [0, 17, -1, 2.5, 3.0, True, False, "3"])
def test_yaml_rejects(value):
    from sac import _engine as E
    with pytest.raises(ValueError, match="buffer.n_step"):
        E.n_step_config(_cfg(value))
    with pytest.raises(ValueError, match="buffer.n_step"):
        E.make_config(4, 2, _cfg(value))


def test_config_field_takes_the_reserved_word():
    """n_step is the struct's last int32 (the former reserved word): layout and size unchanged, and the library agrees."""
    from sac import _engine as E
    assert E.SacxConfig.n_step.offset == E.SacxConfig.agent_id_base.offset + 4
    assert C.sizeof(E.SacxConfig) == 200 == E.SacxConfig.n_step.offset + 4
    lib = E.load()
    assert lib.sacx_sizeof_config() == C.sizeof(E.SacxConfig)


@pytest.mark.parametrize("n,ok", [(0, True), (1, True), (16, True), (17, False), (-1, False)])
def test_library_validates_n_step(n, ok):
    """sacx_agent_arena_floats runs the same validation as sacx_agent_create (no device needed): 0..16, 0 meaning 1."""
    from sac import _engine as E
    lib = E.load()
    cfg = E.make_config(4, 2, _cfg())
    cfg.n_step = n
    out = C.c_int64()
    rc = lib.sacx_agent_arena_floats(C.byref(cfg), C.byref(out))
    if ok:
        assert rc == E.SACX_OK and out.value > 0
    else:
        assert rc == E.SACX_ERR_INVALID
        assert b"n_step" in lib.sacx_last_error()


# ---------------------------------------------------------------------------------------------- the fold, hand-computed
R8 = np.array([1.0, 2.0, 4.0, 8.0, 16.0, 32.0, 64.0, 128.0], dtype=np.float32)


def _d(*terminals, L=8):
    d = np.zeros(L, dtype=np.float32)
    d[list(terminals)] = 1.0
    return d


@pytest.mark.parametrize("name,d,j,n,m,R,d_eff", [
    # gamma = 0.5: every term is exact in float32, so float32 and float64 agree exactly
    ("no terminal", _d(), 1, 3, 3, 2 + 0.5 * 4 + 0.25 * 8, 1 - 0.25),
    ("terminal at offset 0", _d(1), 1, 3, 1, 2.0, 1.0),
    ("terminal in the middle", _d(2), 1, 4, 2, 2 + 0.5 * 4, 1.0),
    ("terminal at the last step", _d(3), 1, 3, 3, 2 + 0.5 * 4 + 0.25 * 8, 1.0),
    ("terminal just past the window", _d(4), 1, 3, 3, 2 + 0.5 * 4 + 0.25 * 8, 1 - 0.25),
    ("ring end inside the window", _d(), 6, 5, 2, 64 + 0.5 * 128, 1 - 0.5),
    ("newest record", _d(), 7, 5, 1, 128.0, 0.0),
    ("n = 1", _d(), 2, 1, 1, 4.0, 0.0),
    ("n = 1 terminal", _d(2), 2, 1, 1, 4.0, 1.0),
    ("n = 16 capped by the ring end", _d(), 0, 16, 8, sum(0.5 ** i * 2.0 ** i for i in range(8)), 1 - 0.5 ** 7),
])
def test_fold_hand_cases(name, d, j, n, m, R, d_eff):
    assert N.window(d, j, n) == m, name
    r32, d32, end = N.fold_f32(R8, d, j, n, 0.5)
    r64, d64, end64 = N.fold_f64(R8, d, j, n, 0.5)
    assert end == end64 == j + m - 1
    assert r32.dtype == np.float32 and d32.dtype == np.float32
    assert float(r32) == R and r64 == R
    assert float(d32) == d_eff and d64 == d_eff


def test_fold_wrapped_ring():
    """A ring of capacity 5 after 7 pushes holds pushes 2..6 (slots 2, 3, 4, 0, 1): the window follows logical order across
    the physical wrap, and the newest record (push 6) cuts it."""
    cap, pushes = 5, 7
    r_push = np.array([10, 20, 30, 40, 50, 60, 70], dtype=np.float32)
    d_push = np.zeros(7, dtype=np.float32)
    slots = np.full(cap, -1)
    for p in range(pushes):
        slots[p % cap] = p
    oldest = pushes - cap
    logical = [slots[(oldest + k) % cap] for k in range(cap)]
    assert logical == [2, 3, 4, 5, 6]
    r, d = r_push[logical], d_push[logical]
    R, de, end = N.fold_f32(r, d, 1, 10, 0.5)                      # pushes 3, 4, 5, 6 -- slots 3, 4, 0, 1
    assert end == 4 and float(R) == 40 + 0.5 * 50 + 0.25 * 60 + 0.125 * 70 and float(de) == 1 - 0.125


def test_fold_low_discount_power_within_one_ulp():
    """gamma^(m-1) below 1/2: 1 - d_eff is within one ulp of the float32 power; at or above 1/2 it is the power exactly."""
    d = _d()
    for gamma, n in ((0.1, 3), (0.3, 5), (0.5, 2), (0.9, 3), (0.99, 16), (0.999, 8), (0.7, 16)):
        _, d_eff, end = N.fold_f32(R8, d, 0, n, gamma)
        m = end + 1
        g = np.float32(1.0)
        for _ in range(m - 1):
            g = np.float32(g * np.float32(gamma))
        back = np.float32(np.float32(1.0) - d_eff)
        if g >= 0.5:
            assert back == g, (gamma, n)
        else:
            assert abs(float(back) - float(g)) <= float(np.spacing(np.float32(0.5))), (gamma, n)


def test_fold_f32_tracks_f64_on_random_rings():
    rng = np.random.default_rng(7)
    for trial in range(200):
        L = int(rng.integers(1, 40))
        r = rng.standard_normal(L).astype(np.float32)
        d = (rng.random(L) < 0.15).astype(np.float32)
        n, j = int(rng.integers(1, 17)), int(rng.integers(0, L))
        gamma = float(np.float32(rng.choice([0.5, 0.9, 0.99, 0.999, 0.3])))
        r32, d32, e32 = N.fold_f32(r, d, j, n, gamma)
        r64, d64, e64 = N.fold_f64(r, d, j, n, gamma)
        assert e32 == e64
        assert abs(float(r32) - r64) <= 1e-5 * (1.0 + np.abs(r[j:e64 + 1]).sum())
        assert abs(float(d32) - d64) <= 1e-6


def test_target_identity():
    """sac_target(R, d_eff) = R + gamma (1 - d_eff)(...) is the n-step target R + gamma^m (1 - d_end)(...)."""
    rng = np.random.default_rng(3)
    r = rng.standard_normal(12)
    for d in (_d(L=12), _d(5, L=12)):
        for j, n, gamma in ((0, 4, 0.99), (3, 3, 0.9), (9, 6, 0.5), (2, 16, 0.999)):
            R, de, end = N.fold_f64(r, d, j, n, gamma)
            g = float(np.float32(gamma))
            tq1, tq2, lp2, alpha = 1.5, 1.25, -0.75, 0.2
            one_step = R + g * (1.0 - de) * (min(tq1, tq2) - alpha * lp2)
            assert abs(one_step - N.target_f64(r, d, j, n, gamma, tq1, tq2, lp2, alpha)) < 1e-12


def test_population_and_data_parallel_carry_n_step():
    """The multi-agent front ends build their engine config through make_config: n_step reaches them unchanged."""
    from sac import _engine as E
    cfg = copy.deepcopy(_cfg(5))
    assert E.make_config(4, 2, cfg, n_agents=8).n_step == 5
    assert E.make_config(4, 2, cfg, dp_world=4, dp_rank=2, batch_size=4).n_step == 5
