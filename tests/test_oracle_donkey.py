"""oracle/donkey_obs.py against the REAL DonkeyVAEEnv methods of the reference (imported here when SAC_REFERENCE_DIR names a
checkout of it; the class needs the simulator only in __init__, so the two methods are called on a bare instance carrying just
the fields they read)."""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest

REF_DIR = os.environ.get("SAC_REFERENCE_DIR", "")
REF = os.path.join(REF_DIR, "DonkeyCarEnv", "donkey_gym", "envs", "vae_env.py")


@pytest.mark.skipif(not REF_DIR or not os.path.exists(REF), reason="reference checkout not present (set SAC_REFERENCE_DIR)")
@pytest.mark.parametrize("z,n_hist,n_stack", [(32, 20, 3), (32, 20, 1), (8, 3, 4)])
def test_oracle_matches_reference_postprocessing(z, n_hist, n_stack, monkeypatch):
    from oracle.donkey_obs import DonkeyObsOracle
    # stub what vae_env.py imports at module level (gymnasium, simulator plumbing, constants): none of it is used by the method
    # under test; the module is loaded under its own dotted name so that its relative imports resolve to the stubs
    here = os.path.dirname(os.path.abspath(__file__))
    try:
        import gymnasium  # noqa: F401
    except ImportError:
        monkeypatch.syspath_prepend(os.path.join(here, "gym_shim"))
        import gymnasium
    if not hasattr(gymnasium, "utils"):
        utils = types.ModuleType("gymnasium.utils")
        utils.seeding = types.SimpleNamespace()
        monkeypatch.setitem(sys.modules, "gymnasium.utils", utils)
        monkeypatch.setattr(gymnasium, "utils", utils, raising=False)
    for name in ("DonkeyCarEnv", "DonkeyCarEnv.config_env", "DonkeyCarEnv.donkey_gym", "DonkeyCarEnv.donkey_gym.core",
                 "DonkeyCarEnv.donkey_gym.core.donkey_proc", "DonkeyCarEnv.donkey_gym.envs", "DonkeyCarEnv.donkey_gym.envs.donkey_sim"):
        m = types.ModuleType(name)
        m.__path__ = []
        monkeypatch.setitem(sys.modules, name, m)
    for k in ("INPUT_DIM", "MIN_STEERING", "MAX_STEERING", "JERK_REWARD_WEIGHT", "MAX_STEERING_DIFF"):
        setattr(sys.modules["DonkeyCarEnv.config_env"], k, 1.0)
    sys.modules["DonkeyCarEnv.donkey_gym.core.donkey_proc"].DonkeyUnityProcess = object
    sys.modules["DonkeyCarEnv.donkey_gym.envs.donkey_sim"].DonkeyUnitySimContoller = object
    spec = importlib.util.spec_from_file_location("DonkeyCarEnv.donkey_gym.envs.vae_env", REF)
    mod = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(mod)
    except Exception as e:  # an import the stubs do not cover
        pytest.skip(f"reference vae_env.py does not import here: {e}")
    env = object.__new__(mod.DonkeyVAEEnv)
    env.n_commands, env.n_command_history, env.n_stack = 2, n_hist, n_stack
    env.command_history = np.zeros((1, 2 * n_hist))
    env.stacked_obs = np.zeros((1, n_stack * (z + 2 * n_hist)), np.float32) if n_stack > 1 else None
    env.jerk_penalty = lambda: 0.0
    ora = DonkeyObsOracle(z, 2, n_hist, n_stack)
    rng = np.random.default_rng(1)
    for t in range(30):
        lat = rng.standard_normal((1, z)).astype(np.float32)
        act = rng.uniform(-1, 1, 2).astype(np.float32)
        done = t % 7 == 6
        got_ref, _, _, _ = env.postprocessing_step(act, lat, 0.5, done, {})
        got = ora.step(lat, act, done)
        assert np.array_equal(np.asarray(got_ref), np.asarray(got)), t
