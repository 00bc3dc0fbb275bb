"""Drop-in surface (SURVEY section 8b), CPU side: every import the reference's callers make resolves against THIS package,
the probe environments behave like the reference's, and the unmodified reference main.py gets as far as constructing the
agent (where this repo, by design, refuses to run without a CUDA device). gymnasium is not installed in the build image:
tests/gym_shim provides the few names the callers touch (harness only)."""
import importlib
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "soft-actor-critic_b200")
SHIM = os.path.join(HERE, "gym_shim")
REF = os.environ.get("SAC_REFERENCE_DIR", "")       # a checkout of ignaschuemer7/soft-actor-critic; tests needing it skip without


@pytest.fixture()
def shim(monkeypatch):
    try:
        import gymnasium  # noqa: F401  (a real installation wins)
    except ImportError:
        monkeypatch.syspath_prepend(SHIM)
    yield
    for m in [m for m in sys.modules if m == "gymnasium" or m.startswith("gymnasium.")]:
        if SHIM in (getattr(sys.modules[m], "__file__", "") or ""):
            del sys.modules[m]
    sys.modules.pop("sac.envs", None)


def test_imports_the_callers_make_resolve(shim):
    """main.py:6-7, sac/agent.py:4-5, the notebooks (SURVEY 8b 'Imports that must resolve')."""
    from sac.agent import SAC  # noqa: F401
    from sac.models import PolicyNetwork, QNetwork  # noqa: F401
    from sac.replay_buffer import ReplayBuffer, Transition  # noqa: F401
    from sac.utils.logger_utils import save_lengths, save_rewards  # noqa: F401
    from sac.random_agent import random_agent_loop  # noqa: F401
    from sac.utils.stable_baseline_params import get_sb3_sac_params  # noqa: F401
    ns = {}
    exec("from sac.envs import *", ns)
    assert {"ConstantRewardEnv", "QuadraticActionRewardEnv", "RandomObsBinaryRewardEnv", "OneDPointMassReachEnv"} <= set(ns)
    spec = importlib.util.find_spec("sac.utils.stable_baseline_logger")           # needs stable_baselines3 to import
    assert spec is not None and spec.origin.startswith(PKG)
    assert importlib.import_module("sac.agent").__file__.startswith(PKG)


def test_sb3_param_mapping(shim):
    from sac.utils.stable_baseline_params import get_sb3_sac_params
    from gpu_helpers import base_config
    from sac.envs import OneDPointMassReachEnv
    cfg = base_config(hidden=(64, 32), act="tanh", auto=True, batch=128)
    p = get_sb3_sac_params(OneDPointMassReachEnv(), cfg, seed=7, env_id="X")
    assert p["ent_coef"] == "auto" and p["target_entropy"] == -1 and p["batch_size"] == 128 and p["seed"] == 7
    assert p["policy_kwargs"]["net_arch"] == {"pi": [64, 32], "qf": [64, 32]} and p["policy_kwargs"]["activation_fn"].__name__ == "Tanh"
    cfg["sac"]["auto_entropy_tuning"] = False
    assert get_sb3_sac_params(OneDPointMassReachEnv(), cfg, 0)["ent_coef"] == cfg["sac"]["alpha"]


@pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "sac", "envs.py")),
                    reason="reference checkout not present (set SAC_REFERENCE_DIR)")
@pytest.mark.parametrize("name,kwargs", [("ConstantRewardEnv", {}), ("ConstantRewardEnv", {"reward": -2.5, "max_steps": 3}),
                                         ("QuadraticActionRewardEnv", {}), ("QuadraticActionRewardEnv", {"target": -0.3, "max_steps": 2}),
                                         ("RandomObsBinaryRewardEnv", {}), ("RandomObsBinaryRewardEnv", {"obs_dim": 7, "max_steps": 4}),
                                         ("OneDPointMassReachEnv", {}), ("OneDPointMassReachEnv", {"goal_pos": -0.4, "max_steps": 9, "dt": 0.5})])
def test_probe_envs_behave_like_the_reference(shim, name, kwargs):
    """Same spaces, observations, rewards, terminated/truncated flags and info dicts as the reference's sac/envs.py on the
    same seeds and action sequences."""
    spec = importlib.util.spec_from_file_location("_reference_envs", os.path.join(REF, "sac", "envs.py"))
    ref_mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_mod)
    import sac.envs as mine_mod
    assert mine_mod.__file__.startswith(PKG)
    a, b = getattr(ref_mod, name)(**kwargs), getattr(mine_mod, name)(**kwargs)
    for sp in ("action_space", "observation_space"):
        sa, sb = getattr(a, sp), getattr(b, sp)
        assert sa.shape == sb.shape and sa.dtype == sb.dtype and np.array_equal(sa.low, sb.low) and np.array_equal(sa.high, sb.high)
    rng = np.random.default_rng(0)
    for ep in range(6):
        oa, ia = a.reset(seed=ep) if ep % 2 == 0 else a.reset()
        ob, ib = b.reset(seed=ep) if ep % 2 == 0 else b.reset()
        assert np.array_equal(oa, ob) and oa.dtype == ob.dtype and ia == ib
        done = False
        while not done:
            act = rng.uniform(-1.5, 1.5, size=1).astype(np.float32)
            ra, rb = a.step(act.copy()), b.step(act.copy())
            assert np.array_equal(ra[0], rb[0]) and ra[1] == rb[1] and ra[2] == rb[2] and ra[3] == rb[3] and ra[4] == rb[4], (ep, ra, rb)
            done = ra[2] or ra[3]


@pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "main.py")),
                    reason="reference checkout not present (set SAC_REFERENCE_DIR)")
def test_unmodified_reference_main_reaches_the_agent_constructor(tmp_path):
    """The reference's `python main.py --config <yaml>` with this package first on PYTHONPATH: the YAML loads, every import
    resolves to this repo, the named probe environment is built, and the run stops exactly where this repo must stop on a
    GPU-less host -- SAC(...) refusing a non-CUDA / absent device (no CPU fallback). On the B200 box the same flow runs to
    'Final average return:' (tests/test_gpu_dropin.py)."""
    import yaml
    from gpu_helpers import base_config
    cfg = base_config(hidden=(32, 32), batch=32, auto=False)
    cfg["logger"]["env_name"] = "OneDPointMassReachEnv"
    cfg["train"]["num_episodes"] = 2
    cfg["train"]["device"] = "cuda"
    path = tmp_path / "cfg.yaml"
    path.write_text(yaml.safe_dump(cfg))
    probe = ("import sys, runpy; import sac.agent, sac.envs; "
             "assert sac.agent.__file__.startswith(%r) and sac.envs.__file__.startswith(%r); "
             "sys.argv = ['main.py', '--config', %r]; runpy.run_path(%r, run_name='__main__')") % (PKG, PKG, str(path), os.path.join(REF, "main.py"))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([PKG, SHIM]), CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True, timeout=300, env=env, cwd=str(tmp_path))
    assert "Configuration loaded:" in p.stdout, p.stdout + p.stderr
    assert p.returncode != 0 and "RuntimeError" in p.stderr and ("CUDA" in p.stderr or "libsacx" in p.stderr), p.stderr[-1500:]
    assert "ModuleNotFoundError" not in p.stderr and "ImportError" not in p.stderr and "NameError" not in p.stderr
