"""-m gpu: population-based training's exploit step (SACPopulation.exploit -> sacx_pbt_copy / pbt_copy_kernel) on the FFMA
population path (SACX_TC_POP=0) and on the tensor-core population path (64 agents x batch 256 = 16 384 rows).

After an exploit every destination holds, in bits, its source's learner state from before the call (parameters, Adam m / v,
targets, the copied scalar fields) and keeps its own update counter, RNG keys, metrics, gradient and batch scratch and ring;
every other agent's arena block and the whole ring are untouched. Records write exactly set_trial's values. Three updates after
an exploit equal three updates of a twin population whose destination was given the same state through the arena views.
"""
import numpy as np
import pytest
import torch

from gpu_helpers import base_config
from helpers import synth_transitions

pytestmark = pytest.mark.gpu

OBS, ACT = 24, 4
CASES = {"ffma": dict(n=6, env={"SACX_TC_POP": "0"}, tc=False), "tc": dict(n=64, env={}, tc=True)}
PAIRS = [(0, 3), (0, 4), (1, 5)]                   # agent 0 feeds two destinations
HYPERS = [None, {"alpha_lr": 7.5e-4, "tau": 0.0123, "gamma": 0.9712345}, {"actor_lr": 1.1e-4, "critic_lr": 2.2e-3, "alpha": 0.37}]


def make_pop(case, auto, monkeypatch):
    from sac.population import SACPopulation
    for k in ("SACX_TC", "SACX_TC_POP", "SACX_TC_MIN_BATCH"):
        monkeypatch.delenv(k, raising=False)
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    n = case["n"]
    cfg = base_config(hidden=(128, 128), batch=256, capacity=600, rng="device", auto=auto, alpha=0.2)
    pop = SACPopulation(OBS, ACT, cfg, n, seeds=[11 + 3 * g for g in range(n)], reference_init=False)
    assert pop.engine.tensor_core()[0] == case["tc"], pop.engine.tensor_core()
    s, a, r, s2, d = (torch.from_numpy(x).cuda() for x in synth_transitions(500, OBS, ACT, 7))
    pop.push_device_all(s, a, r, s2, d.float())
    rng = np.random.default_rng(5)
    pop.set_trials([{"alpha": float(rng.uniform(0.05, 0.5)), "alpha_lr": float(rng.uniform(1e-4, 1e-3)),
                     "actor_lr": float(rng.uniform(1e-4, 1e-3)), "critic_lr": float(rng.uniform(1e-4, 1e-3)),
                     "tau": float(rng.uniform(0.001, 0.05)), "gamma": float(rng.uniform(0.9, 0.999))} for _ in range(n)])
    pop.update(2)                                   # agents differ in everything: weights, Adam state, counters, scalars
    torch.cuda.synchronize()
    return pop


def _words(eng):
    """int32 words of every agent's arena block: [n_agents, stride]."""
    return eng.arena.view(torch.int32).view(eng.n_agents, eng.stride).clone()


def _span(eng, name):
    off, _, cols, _, _ = eng.layout[name]
    return off, off + cols


def _scal_words(eng):
    """(copied, kept) word indices of the scalar block, from the layout's named views."""
    o = {k: eng.layout[k][0] for k in ("scal.log_alpha", "scal.updates", "scal.alpha_lr", "scal.metrics", "scal.lr", "scal.rng_agent")}
    n = eng.layout["scalars"][2]
    kept = set(range(o["scal.updates"], o["scal.alpha_lr"])) | set(range(o["scal.metrics"], o["scal.lr"])) | \
        set(range(o["scal.rng_agent"], n))
    return [w for w in range(n) if w not in kept], sorted(kept)


def _state_words(eng):
    """Word ranges of the learner state: the scalar block is handled word by word."""
    return [_span(eng, n) for n in ("block.params", "block.m", "block.v", "block.targets")]


def _expected_scalars(eng, rec_vals, auto):
    """{view name: expected python value} of a record, the way set_trial writes it."""
    out = {}
    for k, v in (rec_vals or {}).items():
        if k == "alpha" and not auto:
            out["scal.log_alpha"] = np.float64(np.log(v))
            out["scal.alpha"] = np.float64(np.float32(v))
            out["scal.alpha_f32"] = np.float32(v)
        elif k == "alpha_lr":
            out["scal.alpha_lr"] = np.float64(v)
        elif k == "actor_lr":
            out["scal.lr[0]"] = np.float64(v)
        elif k == "critic_lr":
            out["scal.lr[1]"] = out["scal.lr[2]"] = np.float64(v)
        elif k == "tau":
            out["scal.tau[0]"] = np.float32(v)
            out["scal.tau[1]"] = np.float32(1.0 - v)
        elif k == "gamma":
            out["scal.gamma"] = np.float32(v)
    return out


def _read_scalar(eng, agent, key):
    name, _, idx = key.partition("[")
    t = eng.view(name, agent).reshape(-1)
    return t[int(idx[:-1]) if idx else 0].item()


def _record_words(eng, rec_vals, auto):
    """Scalar-block words a record writes (they equal the record, not the source)."""
    words = set()
    for key in _expected_scalars(eng, rec_vals, auto):
        name, _, idx = key.partition("[")
        off, _, _, _, dtype = eng.layout[name]
        width = 2 if dtype in (1, 2) else 1
        i = int(idx[:-1]) if idx else 0
        words |= set(range(off + i * width, off + (i + 1) * width))
    return words


def check_exploit(pop, pairs, hypers, auto):
    eng = pop.engine
    before = _words(eng)
    ring_before = pop.ring._store.clone()
    pop.exploit(pairs, hypers)
    torch.cuda.synchronize()
    after = _words(eng)
    assert torch.equal(pop.ring._store, ring_before), "a ring changed"
    dsts = {d: (s, (hypers or [None] * len(pairs))[i]) for i, (s, d) in enumerate(pairs)}
    copied, kept = _scal_words(eng)
    spans = _state_words(eng)
    in_state = torch.zeros(eng.stride, dtype=torch.bool, device=after.device)
    for a, b in spans:
        in_state[a:b] = True
    in_state[: eng.layout["scalars"][2]] = True
    for ag in range(eng.n_agents):
        if ag not in dsts:
            assert torch.equal(after[ag], before[ag]), f"agent {ag} is not a destination but changed"
            continue
        src, rec = dsts[ag]
        for a, b in spans:
            assert torch.equal(after[ag, a:b], before[src, a:b]), (ag, a, b)
        assert torch.equal(after[ag][~in_state], before[ag][~in_state]), f"agent {ag}: scratch / gradients changed"
        rec_words = _record_words(eng, rec, auto)
        for w in copied:
            if w not in rec_words:
                assert after[ag, w] == before[src, w], (ag, "scalar word", w)
        for w in kept:
            assert after[ag, w] == before[ag, w], (ag, "kept scalar word", w)
        for key, want in _expected_scalars(eng, rec, auto).items():
            got = _read_scalar(eng, ag, key)
            assert type(want)(got).tobytes() == want.tobytes(), (ag, key, got, want)


@pytest.mark.parametrize("path", list(CASES))
@pytest.mark.parametrize("auto", [True, False], ids=["auto_alpha", "fixed_alpha"])
def test_exploit_copies_state_and_keeps_the_rest(path, auto, monkeypatch):
    pop = make_pop(CASES[path], auto, monkeypatch)
    check_exploit(pop, PAIRS, HYPERS, auto)
    if auto:                                        # the temperature travels with the state; a record never writes it
        assert pop.engine.view("scal.log_alpha", 5).item() == pop.engine.view("scal.log_alpha", 1).item()
    check_exploit(pop, [(5, 2)], None, auto)        # a former destination as a source, no records


def test_exploit_refusals(monkeypatch):
    from sac import _engine as E
    pop = make_pop(CASES["ffma"], False, monkeypatch)
    eng = pop.engine
    before = _words(eng)
    for pairs, hypers in (([(0, 6)], None), ([(-1, 2)], None), ([(0, 1), (2, 1)], None), ([(0, 1), (1, 2)], None),
                          ([(3, 3)], None), ([(0, 1)], [{"tau": 0.0}]), ([(0, 1)], [{"actor_lr": -1.0}]),
                          ([(0, 1)], [{"gamma": float("nan")}])):
        with pytest.raises(ValueError):
            pop.exploit(pairs, hypers)
    bad = E.SacxPbtRecord()
    bad.set, bad.gamma = E.PBT_GAMMA, -0.5
    with pytest.raises(ValueError, match="gamma"):                 # the library's own check, before any device work
        eng.pbt_copy([0], [1], [bad])
    with pytest.raises(ValueError, match="out of range"):
        eng.pbt_copy([0], [6])
    with pytest.raises(ValueError, match="both a source and a destination"):
        eng.pbt_copy([0, 1], [1, 2])
    with pytest.raises(ValueError, match="slot"):
        eng.pbt_unpack(torch.zeros(eng.pbt_state_floats(), device=eng.device), [1], [0])
    torch.cuda.synchronize()
    assert torch.equal(_words(eng), before), "a refused call changed the arena"


def test_exploit_refuses_a_temperature_record_with_auto_tuning(monkeypatch):
    from sac import _engine as E
    pop = make_pop(CASES["ffma"], True, monkeypatch)
    r = E.SacxPbtRecord()
    r.set, r.alpha, r.alpha_f32, r.log_alpha = E.PBT_ALPHA, 0.3, 0.3, float(np.log(0.3))
    with pytest.raises(ValueError, match="auto_entropy_tuning"):
        pop.engine.pbt_copy([0], [1], [r])


def test_pack_unpack_equals_copy(monkeypatch):
    pop = make_pop(CASES["ffma"], False, monkeypatch)
    eng = pop.engine
    twin_words = _words(eng)
    buf = torch.empty((2, eng.pbt_state_floats()), device=eng.device)
    eng.pbt_pack([1, 0], buf)
    eng.pbt_unpack(buf, [1, 0, 0], [3, 4, 5])
    torch.cuda.synchronize()
    unpacked = _words(eng)
    eng.arena.view(torch.int32).copy_(twin_words.view(-1))
    eng.pbt_copy([0, 1, 1], [3, 4, 5])
    torch.cuda.synchronize()
    assert torch.equal(_words(eng), unpacked)


@pytest.mark.parametrize("path", list(CASES))
@pytest.mark.parametrize("auto", [True, False], ids=["auto_alpha", "fixed_alpha"])
def test_three_updates_after_exploit_equal_a_twin_given_the_state_by_views(path, auto, monkeypatch):
    pop = make_pop(CASES[path], auto, monkeypatch)
    twin = make_pop(CASES[path], auto, monkeypatch)
    assert torch.equal(_words(pop.engine), _words(twin.engine)), "two populations built alike differ"
    src, dst, rec = 2, 4, {"alpha": 0.31, "critic_lr": 1.7e-3, "tau": 0.02}
    pop.exploit([(src, dst)], [rec])
    e = twin.engine
    for name in ("block.params", "block.m", "block.v", "block.targets"):
        e.view(name, dst).copy_(e.view(name, src))
    for name in ("scal.log_alpha", "scal.alpha_m", "scal.alpha_v", "scal.alpha", "scal.step", "scal.alpha_lr", "scal.alpha_f32",
                 "scal.lr", "scal.gamma", "scal.tau"):
        e.view(name, dst).copy_(e.view(name, src))
    w = e.arena.view(torch.int32)                    # Adam bias corrections: the words between alpha_f32 and the metrics
    a, b = e.layout["scal.alpha_f32"][0] + 1, e.layout["scal.metrics"][0]
    w[dst * e.stride + a: dst * e.stride + b].copy_(w[src * e.stride + a: src * e.stride + b])
    if not auto:
        e.view("scal.log_alpha", dst).fill_(float(np.log(0.31)))
        e.view("scal.alpha", dst).fill_(float(np.float32(0.31)))
        e.view("scal.alpha_f32", dst).fill_(float(np.float32(0.31)))
    e.view("scal.lr", dst)[1:] = 1.7e-3
    e.view("scal.tau", dst).reshape(-1).copy_(torch.tensor([np.float32(0.02), np.float32(1.0 - 0.02)]))
    torch.cuda.synchronize()
    assert torch.equal(_words(pop.engine), _words(e)), "exploit and the view-built state differ before the updates"
    pop.update(3)
    twin.update(3)
    torch.cuda.synchronize()
    assert torch.equal(_words(pop.engine), _words(e)), "three updates after the exploit differ from the twin's"
    assert pop.engine.view("scal.updates", dst).item() == pop.engine.view("scal.updates", src).item()


def _pbt_run(out):
    import os
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    shim = os.path.join(here, "gym_shim")
    try:
        import gymnasium  # noqa: F401
    except ImportError:
        sys.path.insert(0, shim)
    from sac.envs import OneDPointMassReachEnv
    from sac.pbt import PBTConfig
    from sac.trials import run_population_pbt
    space = {"sac": {"alpha": {"type": "loguniform", "low": 0.005, "high": 0.05},
                     "actor_lr": {"type": "loguniform", "low": 1e-4, "high": 1e-3},
                     "critic_lr": {"type": "loguniform", "low": 1e-4, "high": 1e-3}}}
    cfg = base_config(hidden=(256, 256), batch=256, auto=False, alpha=0.02, rng="device")
    cfg["train"].update(warming_steps=1000, device="cuda")
    return run_population_pbt(cfg, space, 8, OneDPointMassReachEnv, PBTConfig(interval_steps=2500, fraction=0.25, seed=3),
                              num_episodes=400, seed=2, out=out)


def test_pbt_driver_end_to_end_on_point_mass():
    """Eight trials on OneDPointMassReachEnv with exploit rounds every 2 500 environment steps: every trial prints its final
    return, at least one PBT line appears, the best trial reaches the drop-in test's band, and a second run prints the same."""
    lines = []
    res = _pbt_run(lines.append)
    finals = [float(l.split(":")[1].strip()) for l in lines if l.startswith("Final average return:")]
    assert len(finals) == 8
    pbt_lines = [l for l in lines if l.startswith("PBT step ")]
    assert pbt_lines and all(" <- trial " in l for l in pbt_lines)
    assert res["best_value"] >= 0.80, (res["best_value"], finals)
    assert any(res["lineage"]) and res["final_trials"] != res["trials"]
    assert any("--- PBT Lineage ---" in l for l in lines)
    again = []
    _pbt_run(again.append)
    assert again == lines
