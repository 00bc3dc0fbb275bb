"""Prioritized replay without a device: YAML validation, the float64 oracle on hand-computed cases, and the C ABI surface."""
import copy
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PER_SYMBOLS = ("sacx_per_create", "sacx_per_destroy", "sacx_per_sample", "sacx_per_update_priorities", "sacx_per_priorities",
               "sacx_per_load_priorities", "sacx_agent_attach_per")


def _cfg(prioritized="absent", rng="device"):
    cfg = {"buffer": {"capacity": 1000}, "train": {"rng": rng, "batch_size": 32, "seed": 0}}
    if prioritized != "absent":
        cfg["buffer"]["prioritized"] = prioritized
    return cfg


def test_yaml_defaults_and_absent_key():
    from sac import _engine as E
    assert E.per_config(_cfg()) is None
    assert E.per_config(_cfg(None)) is None
    assert E.per_config(_cfg({})) == {"alpha": 0.6, "beta": 0.4, "beta_steps": 0, "eps": 1e-6}
    got = E.per_config(_cfg({"alpha": 0.7, "beta_steps": 1000}))
    assert got == {"alpha": 0.7, "beta": 0.4, "beta_steps": 1000, "eps": 1e-6}


@pytest.mark.parametrize("bad", [{"alpha": -0.1}, {"beta": -0.01}, {"beta": 1.5}, {"eps": 0.0}, {"eps": -1e-6},
                                 {"beta_steps": -1}, {"beta_steps": 2.5}, {"gamma": 1.0}, [0.6]])
def test_yaml_bad_ranges_raise(bad):
    from sac import _engine as E
    with pytest.raises(ValueError):
        E.per_config(_cfg(bad))


def test_yaml_host_rng_and_population_raise():
    from sac import _engine as E
    from sac.population import DataParallelSAC, SACPopulation
    with pytest.raises(ValueError):
        E.per_config(_cfg({}, rng="host"))
    cfg = _cfg({})
    with pytest.raises(ValueError):
        SACPopulation(4, 2, cfg, n_agents=2)
    with pytest.raises(ValueError):
        DataParallelSAC(4, 2, copy.deepcopy(cfg), global_batch=64)


def test_oracle_stratified_sampling_hand_case():
    from oracle import per_numpy as P
    p = np.array([1.0, 0.0, 3.0, 2.0, 0.0, 4.0])          # prefix sums 1 1 4 6 6 10
    # B = 5 strata of width 2: u = 0.5, 2.5, 4.5, 6.5, 8.5
    u = P.strata_u(np.full(5, 0.25), p.sum())
    assert np.allclose(u, [0.5, 2.5, 4.5, 6.5, 8.5])
    assert P.sample(p, u).tolist() == [0, 2, 3, 5, 5]
    # edge draws: u = 0 takes the first nonzero slot, u at or past the total clamps to the last slot with p > 0
    assert P.sample(p, [0.0, 1.0, 10.0, 10.5]).tolist() == [0, 2, 5, 5]
    assert P.sample(np.array([2.0, 5.0, 0.0, 0.0]), [7.0]).tolist() == [1]


def test_oracle_weights_and_priorities():
    from oracle import per_numpy as P
    p = np.array([1.0, 0.0, 4.0, 2.0])
    w = P.weights(p, [1.0, 4.0, 2.0], 0.5)
    assert np.allclose(w, [1.0, 0.5, 2 ** -0.5])
    assert np.all(P.weights(p, [4.0], 0.0) == 1.0)
    d = P.td_delta([1.0, 0.0], [3.0, -2.0], [2.0, 1.0])
    assert np.allclose(d, [1.0, 2.0])
    assert np.allclose(P.priority(d, 0.5, 1e-6), np.sqrt(d + 1e-6))
    assert np.all(P.priority(d, 0.0, 1e-6) == 1.0)
    leaves, pmax = P.write_back(np.zeros(4), [1, 3, 1], [5.0, 2.0, 3.0], 1.0)
    assert leaves.tolist() == [0.0, 3.0, 0.0, 2.0] and pmax == 5.0          # highest row wins; p_max over every row
    assert P.logical_to_slot([0, 1, 4], pushes=7, capacity=5).tolist() == [2, 3, 1]


def test_oracle_beta_schedule():
    from oracle import per_numpy as P
    assert P.beta_at(0, 0.4, 0) == 0.4 and P.beta_at(10 ** 9, 0.4, 0) == 0.4
    assert P.beta_at(0, 0.4, 100) == 0.4
    assert abs(P.beta_at(50, 0.4, 100) - 0.7) < 1e-15
    assert P.beta_at(100, 0.4, 100) == 1.0 and P.beta_at(1000, 0.4, 100) == 1.0


def test_per_symbols_in_header_binding_and_library():
    import __graft_entry__ as g
    g.build()
    from sac import _engine as E
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "sacx.h")).read(), flags=re.S)
    lib = E.load()
    for name in PER_SYMBOLS:
        assert re.search(r"\b%s\s*\(" % name, src), name
        assert name in E.SYMBOLS, name
        assert hasattr(lib, name), name


def test_per_create_refuses_bad_arguments_without_a_device():
    """Argument checks come before any device work: bad ranges and null handles are SACX_ERR_INVALID."""
    import ctypes as C
    from sac import _engine as E
    lib = E.load()
    h = C.c_void_p()
    assert lib.sacx_per_create(None, 0.6, 0.4, 0, 1e-6, 256, C.byref(h)) == E.SACX_ERR_INVALID
    assert lib.sacx_per_sample(None, 256, 0.4, None, 0, 0, None, None) == E.SACX_ERR_INVALID
    assert lib.sacx_per_update_priorities(None, None, None, 4) == E.SACX_ERR_INVALID
    assert lib.sacx_agent_attach_per(None, None) == E.SACX_ERR_INVALID
