"""-m gpu: n-step returns (buffer.n_step) folded into the batch gather of every update path.

- The fold in bits: batch.r / batch.d / the state columns of batch.s2a / batch.idx equal oracle/nstep_numpy.py's float32
  restatement exactly, on every path the config selects, for indices aimed at the newest records and at terminals at every
  offset of the window (idx_ext) and for the device's own draws.
- The update is the one-step update of the folded ring: an n-step update on ring X leaves the whole arena bit-identical to a
  one-step update with the same indices and normals on ring X', whose record j is (s[j], a[j], R, s2[j+m-1], d_eff).
- Semantics: out.y against the float64 n-step target built from the engine's own tq1, tq2, logpi_next and alpha.
- n_step: 1 and an absent key are the same engine, bit for bit.
"""
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_helpers import FakeEnv, base_config, load_nets
from helpers import rel_l2
from oracle import nstep_numpy as N
from test_gpu_parity import _random_nets
from update_oracle import SWITCHES, per_slots

pytestmark = pytest.mark.gpu

F32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
D = (256, 256)
NS = (2, 3, 5, 16)


def _bits(name, got, want):
    got = np.ascontiguousarray(got.detach().cpu().numpy() if torch.is_tensor(got) else got, dtype=F32)
    want = np.ascontiguousarray(want, dtype=F32)
    assert got.shape == want.shape, (name, got.shape, want.shape)
    bad = np.flatnonzero(got.view(np.uint32).ravel() != want.view(np.uint32).ravel())
    assert bad.size == 0, f"{name}: {bad.size} elements differ, first at {bad[0]}: {got.ravel()[bad[0]]!r} != {want.ravel()[bad[0]]!r}"


def _ring_data(rng, n_push, O, A):
    s = rng.standard_normal((n_push, O)).astype(F32)
    s2 = rng.standard_normal((n_push, O)).astype(F32)
    a = rng.uniform(-1, 1, (n_push, A)).astype(F32)
    r = rng.standard_normal(n_push).astype(F32)
    d = (rng.random(n_push) < 0.2).astype(F32)
    return s, a, r, s2, d


def _push(rb, data, cap, agent=0):
    for lo in range(0, len(data[0]), cap // 2):
        rb.push_batch(*(x[lo: lo + cap // 2] for x in data), agent=agent)


def _engine(monkeypatch, O, A, B, n_step, env=None, n_agents=1, hp=D, hq=D, seed=0, gammas=None, dp=None):
    from sac.engine import UpdateEngine
    for k in SWITCHES + ("SACX_TC_POP",):
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    cfg = base_config(hidden=hp, q_hidden=hq, batch=B, seed=seed, rng="device")
    if n_step != "absent":
        cfg["buffer"]["n_step"] = n_step
    kw = dict(dp_world=dp[0], dp_rank=dp[1], batch_size=B // dp[0]) if dp else {}
    eng = UpdateEngine(O, A, cfg, n_agents=n_agents, **kw)
    sds = _random_nets(O, A, hp, hq, seed=seed, scale=0.15)
    for ag in range(n_agents):
        load_nets(eng, sds, agent=ag)
    eng.reset_state()
    for ag, g in enumerate(gammas or []):
        eng.view("scal.gamma", ag).fill_(float(g))
    return eng


def _ring(O, A, cap, n_agents=1, seed=1, wrap=True, per=None):
    """A wrapped ring (oldest slot != 0) per agent; returns (buffer, [logical (s, a, r, s2, d) per agent], pushes)."""
    from sac.replay_buffer import PrioritizedReplayBuffer, ReplayBuffer
    rng = np.random.default_rng(seed)
    n_push = cap + cap // 3 + 7 if wrap else cap - 5
    rb = PrioritizedReplayBuffer(cap, O, A, **per) if per else ReplayBuffer(cap, O, A, n_agents=n_agents)
    logical = []
    for ag in range(n_agents):
        data = _ring_data(rng, n_push, O, A)
        _push(rb, data, cap, agent=ag)
        first = max(n_push - cap, 0)
        logical.append(tuple(x[first:] for x in data))
    return rb, logical, n_push


def _aimed_indices(d, n, B, rng):
    """Logical indices whose window ends at a terminal at every offset 0..n-1, the n newest records, then random fill."""
    L = len(d)
    out = list(range(max(L - n, 0), L))
    for k in range(n):
        hits = [j for j in range(L - k) if d[j + k] != 0 and not d[j: j + k].any()]
        out += hits[:2]
    out = out[:B]
    out += rng.integers(0, L, B - len(out)).tolist()
    return np.array(out, dtype=np.int64)


def _check_batch(eng, logical, n, gamma, agent=0, idx=None):
    s, a, r, s2, d = logical
    O, A = s.shape[1], a.shape[1]
    got_idx = eng.view("batch.idx", agent).cpu().numpy().reshape(-1)
    if idx is not None:
        assert np.array_equal(got_idx, idx)
    R, De, end = N.fold_batch_f32(r, d, got_idx, n, gamma)
    _bits("batch.r", eng.view("batch.r", agent).reshape(-1), R)
    _bits("batch.d", eng.view("batch.d", agent).reshape(-1), De)
    _bits("batch.s2a states", eng.view("batch.s2a", agent)[:, :O], s2[end])
    _bits("batch.sa states", eng.view("batch.sa", agent)[:, :O], s[got_idx])
    _bits("batch.sa actions", eng.view("batch.sa", agent)[:, O:O + A], a[got_idx])
    return got_idx


# id: (obs, act, batch, env, expected path, tensor core)
PATHS = {
    "rowpar": (24, 4, 256, {}, "rowpar", False),
    "rowpar-groups1-cpasync": (24, 4, 256, {"SACX_RP_GROUPS": "1", "SACX_RP_TMA": "0"}, "rowpar", False),
    "rowpar-obs60": (60, 6, 200, {}, "rowpar", False),                           # 8-column gather body
    "ffma32": (24, 4, 256, {"SACX_ROWPAR": "0"}, "tiles", False),
    "ffma64": (24, 4, 1024, {}, "tiles", False),
    "tc": (24, 4, 256, {"SACX_TC_MIN_BATCH": "256"}, "tiles", True),
    "tc-no-rows": (24, 4, 256, {"SACX_TC_MIN_BATCH": "256", "SACX_TC_ROWS": "0"}, "tiles", True),
}


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("path", list(PATHS))
def test_fold_bits_single_agent(path, n, monkeypatch):
    O, A, B, env, kind, tc = PATHS[path]
    eng = _engine(monkeypatch, O, A, B, n, env)
    assert eng.path()[0] == kind and eng.tensor_core()[0] == tc, (eng.path(), eng.tensor_core())
    cap = max(3 * B, 600)
    rb, (lg,), _ = _ring(O, A, cap, seed=n)
    eng.attach_ring(rb)
    rng = np.random.default_rng(n)
    idx = _aimed_indices(lg[4], n, B, rng)
    eng.update(torch.as_tensor(idx).cuda(), None, None, 1)
    gamma = float(eng.view("scal.gamma").item())
    _check_batch(eng, lg, n, gamma, idx=idx)
    eng.update(None, None, None, 1)                                           # the device's own draw
    _check_batch(eng, lg, n, gamma)
    assert (eng.tensor_core()[2] > 0) == tc


@pytest.mark.parametrize("tc", [False, True], ids=["ffma", "tc"])
def test_fold_bits_population_per_agent_gamma(tc, monkeypatch):
    """Population of 4 agents with their own discount trials (sacx gathers each agent's ring with its own gamma)."""
    O, A, B, n = 24, 4, 256, 5
    gammas = (0.5, 0.999, 0.9, 0.99)
    env = {"SACX_TC_MIN_BATCH": "256"} if tc else {"SACX_TC_POP": "0"}
    eng = _engine(monkeypatch, O, A, B, n, env, n_agents=4, gammas=gammas)
    assert eng.tensor_core()[0] == tc
    rb, lgs, _ = _ring(O, A, 900, n_agents=4, seed=7)
    eng.attach_ring(rb)
    rng = np.random.default_rng(3)
    idx = np.stack([_aimed_indices(lg[4], n, B, rng) for lg in lgs])
    eng.update(torch.as_tensor(idx[None]).cuda(), None, None, 1)
    for ag in range(4):
        _check_batch(eng, lgs[ag], n, gammas[ag], agent=ag, idx=idx[ag])
    eng.update(None, None, None, 1)
    for ag in range(4):
        _check_batch(eng, lgs[ag], n, gammas[ag], agent=ag)


@pytest.mark.parametrize("world", [1, 4, 8])
def test_fold_bits_data_parallel_ranks(world, monkeypatch):
    """Emulated data-parallel ranks: each gathers its rows of the global batch (sample_batch: the plan DataParallelSAC uses)."""
    O, A, B, n = 24, 4, 512, 3
    rb, (lg,), _ = _ring(O, A, 1600, seed=11)
    rng = np.random.default_rng(5)
    idx = _aimed_indices(lg[4], n, B, rng)
    drawn = []
    for rank in range(world):
        eng = _engine(monkeypatch, O, A, B, n, dp=(world, rank))
        eng.attach_ring(rb)
        b = B // world
        mine = idx[rank * b:(rank + 1) * b]
        eng.sample_batch(torch.as_tensor(mine).cuda())
        _check_batch(eng, lg, n, 0.99, idx=mine)
        eng.sample_batch(None)
        drawn.append(_check_batch(eng, lg, n, 0.99))
    drawn = np.concatenate(drawn)
    assert len(np.unique(drawn)) == B                                          # one bijection over the global batch


def _per_engine(monkeypatch, n):
    O, A, B, cap = 24, 4, 256, 900
    per = dict(alpha=0.6, beta=0.4, beta_steps=1000, eps=1e-6)
    eng = _engine(monkeypatch, O, A, B, n)
    rb, (lg,), pushes = _ring(O, A, cap, seed=13, per=per)
    eng.attach_ring(rb)
    eng.attach_per(rb)
    return eng, rb, lg, pushes, cap, per


@pytest.mark.parametrize("n", [3, 16])
def test_prioritized_replay_folds_and_writes_back_nstep_delta(n, monkeypatch):
    """The tree picks j, the gather folds; the deferred write-back holds (delta + eps)^alpha with delta from the n-step y."""
    from oracle import per_numpy as P
    eng, rb, lg, pushes, cap, per = _per_engine(monkeypatch, n)
    eng.update(None, None, None, 1)
    idx = _check_batch(eng, lg, n, 0.99)
    q1, q2, y = (eng.view(v).cpu().numpy().ravel() for v in ("out.q1", "out.q2", "out.y"))
    pr = P.priority(P.td_delta(q1, q2, y), float(F32(per["alpha"])), float(F32(per["eps"])))
    slots = per_slots(pushes, cap, len(lg[0]))[idx]
    leaves, _ = rb.slot_priorities()
    leaves = leaves.cpu().numpy()
    last = {int(s): k for k, s in enumerate(slots)}
    ss, ks = np.array(list(last)), np.array(list(last.values()))
    err = float(np.max(np.abs(leaves[ss] - pr[ks]) / pr[ks]))
    assert err < 2e-6, err


def _target_vs_f64(eng, lg, n, gamma, alpha, idx):
    s, a, r, s2, d = lg
    tq1, tq2, lp2, y = (eng.view(v).cpu().numpy().ravel().astype(np.float64)
                        for v in ("out.tq1", "out.tq2", "out.logpi_next", "out.y"))
    ref = np.array([N.target_f64(r, d, int(j), n, gamma, tq1[k], tq2[k], lp2[k], alpha) for k, j in enumerate(idx)])
    return rel_l2(y, ref)


EQUIV = {"rowpar": PATHS["rowpar"], "ffma32": PATHS["ffma32"], "ffma64": PATHS["ffma64"], "tc": PATHS["tc"]}


@pytest.mark.parametrize("n", [3, 16])
@pytest.mark.parametrize("path", list(EQUIV))
def test_update_equals_one_step_update_of_folded_ring(path, n, monkeypatch):
    from sac.replay_buffer import ReplayBuffer
    O, A, B, env, kind, tc = EQUIV[path]
    cap = max(3 * B, 600)
    eng_n = _engine(monkeypatch, O, A, B, n, env)
    eng_1 = _engine(monkeypatch, O, A, B, "absent", env)
    assert eng_n.path()[0] == eng_1.path()[0] == kind and eng_n.tensor_core()[0] == tc
    rb, (lg,), _ = _ring(O, A, cap, seed=21 + n)
    s, a, r, s2, d = lg
    L = len(r)
    R, De, end = N.fold_batch_f32(r, d, np.arange(L), n, 0.99)
    folded = ReplayBuffer(cap, O, A)
    _push(folded, (s, a, R, s2[end], De), cap)
    eng_n.attach_ring(rb)
    eng_1.attach_ring(folded)
    rng = np.random.default_rng(n)
    idx = torch.as_tensor(_aimed_indices(d, n, B, rng)).cuda()
    e1 = torch.as_tensor(rng.standard_normal((B, A)).astype(F32)).cuda()
    e2 = torch.as_tensor(rng.standard_normal((B, A)).astype(F32)).cuda()
    alpha = float(eng_n.view("scal.alpha_f32").item())
    for eng in (eng_n, eng_1):
        eng.update(idx, e1, e2, 1)
    torch.cuda.synchronize()
    assert torch.equal(eng_n.arena.view(torch.int32), eng_1.arena.view(torch.int32)), "arenas differ"
    assert eng_n.metrics() == eng_1.metrics()
    e = _target_vs_f64(eng_n, lg, n, 0.99, alpha, idx.cpu().numpy())
    assert e < 2e-5, e


N1 = {"rowpar": PATHS["rowpar"], "ffma32": PATHS["ffma32"], "ffma64": PATHS["ffma64"],
      "tc": (24, 4, 4096, {}, "tiles", True)}


@pytest.mark.parametrize("path", list(N1))
def test_n_step_one_is_the_absent_key(path, monkeypatch):
    O, A, B, env, kind, tc = N1[path]
    engs = [_engine(monkeypatch, O, A, B, v, env) for v in (1, "absent")]
    rb, _, _ = _ring(O, A, 3 * B, seed=2)
    for eng in engs:
        assert eng.path()[0] == kind and eng.tensor_core()[0] == tc
        eng.attach_ring(rb)
        eng.update(None, None, None, 1)
    torch.cuda.synchronize()
    assert torch.equal(engs[0].arena.view(torch.int32), engs[1].arena.view(torch.int32))
    assert engs[0].metrics() == engs[1].metrics()


@pytest.mark.parametrize("rng_mode", ["host", "device"])
def test_sac_sample_batch_is_the_training_batch(rng_mode, monkeypatch):
    """SAC.sample_batch with n_step > 1 returns the folded batch: host RNG from the reference's index stream, device RNG the
    draw the next training_step makes."""
    from sac.agent import SAC
    from sac.replay_buffer import sample_range
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    O, A, B, n = 8, 2, 64, 4
    cfg = base_config(hidden=(64, 64), batch=B, capacity=500, rng=rng_mode)
    cfg["buffer"]["n_step"] = n
    agent = SAC(FakeEnv(O, A), cfg)
    rng = np.random.default_rng(0)
    s, a, r, s2, d = _ring_data(rng, 700, O, A)
    for k in range(700):
        agent.store_transition(s[k], a[k], float(r[k]), s2[k], bool(d[k]))
    lg = tuple(x[200:] for x in (s, a, r, s2, d))
    state = random.getstate()
    t = agent.sample_batch()
    if rng_mode == "host":
        random.setstate(state)
        idx = np.array(sample_range(500, B), dtype=np.int64)
    else:
        idx = agent.engine.view("batch.idx").cpu().numpy().copy()
        agent.training_step()
        assert np.array_equal(agent.engine.view("batch.idx").cpu().numpy(), idx)
    R, De, end = N.fold_batch_f32(lg[2], lg[4], idx, n, 0.99)
    _bits("state", t.state, lg[0][idx])
    _bits("action", t.action, lg[1][idx])
    _bits("reward", t.reward, R)
    _bits("next_state", t.next_state, lg[3][end])
    _bits("done", t.done, De)


def test_main_process_learns_point_mass_with_n_step_returns(tmp_path):
    import yaml
    from test_gpu_per import _pythonpath
    cfg = base_config(hidden=(256, 256), batch=256, auto=False, alpha=0.02, rng="device")
    cfg["train"].update(warming_steps=1000, num_episodes=400, device="cuda")
    cfg["logger"].update(env_name="OneDPointMassReachEnv", enabled=False)
    cfg["buffer"]["n_step"] = 3
    path = tmp_path / "cfg.yaml"
    path.write_text(yaml.safe_dump(cfg))
    p = subprocess.run([sys.executable, os.path.join(HERE, "run_main_like_reference.py"), "--config", str(path)],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, PYTHONPATH=_pythonpath()), cwd=str(tmp_path))
    assert p.returncode == 0, p.stderr[-3000:]
    final = None
    for line in reversed(p.stdout.strip().split("\n")):
        if "Final average return:" in line:
            final = float(line.split(":")[1].strip())
            break
    assert final is not None, p.stdout[-2000:]
    assert final >= 0.80, f"last-100 average return {final} with 3-step returns"
