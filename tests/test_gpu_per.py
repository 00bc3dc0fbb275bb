"""-m gpu: prioritized experience replay on the device ring (sacx_per_*, PrioritizedReplayBuffer, buffer.prioritized).

Exactness tests use integer priorities (exact float32 prefix sums): either loaded directly (load_slot_priorities) or written
back with alpha = 1, eps = 0.5 and td = n + 0.5, so that every tree sum is an exact integer and the device's choice of slot
must equal the float64 oracle's searchsorted (oracle/per_numpy.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_helpers import FakeEnv, base_config
from helpers import rel_l2, synth_transitions

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _pythonpath():
    """The package, and the gymnasium stand-in of tests/gym_shim unless a real gymnasium is installed (another test may already
    have put the stand-in on this process's path)."""
    shim = os.path.join(HERE, "gym_shim")
    paths = [os.path.join(os.path.dirname(HERE), "soft-actor-critic_b200")]
    try:
        import gymnasium
        if os.path.abspath(gymnasium.__file__).startswith(shim + os.sep):
            paths.append(shim)
    except ImportError:
        paths.append(shim)
    return os.pathsep.join(paths)


def _weighted_port(obs, act, cfg, capacity):
    """TorchPortSAC (the reference update in torch, oracle/torch_port.py) with the critic loss of prioritized replay,
    mean(w (q - y)^2); the actor and temperature steps stay unweighted. The other statements are those of
    TorchPortSAC.update_from_batch."""
    from oracle.torch_port import TorchPortSAC

    class WeightedPort(TorchPortSAC):
        def update_from_batch(self, s, a, r, s2, d, eps1, eps2, weights):
            gamma, tau = self.cfg["sac"]["gamma"], self.cfg["sac"]["tau"]
            with torch.no_grad():
                alpha = self.alpha.detach()
                a2, lp2 = self.sample_action(s2, eps1)
                minq = torch.min(self._q(self.q1t, s2, a2), self._q(self.q2t, s2, a2))
                y = r + gamma * (1 - d) * (minq - alpha * lp2)
            q1v, q2v = self._q(self.q1, s, a), self._q(self.q2, s, a)
            w = torch.as_tensor(weights, dtype=q1v.dtype).reshape(q1v.shape)
            l1 = (w * (q1v - y) ** 2).mean()
            l2 = (w * (q2v - y) ** 2).mean()
            self.opt_q1.zero_grad()
            l1.backward()
            self.opt_q1.step()
            self.opt_q2.zero_grad()
            l2.backward()
            self.opt_q2.step()
            an, lp = self.sample_action(s, eps2)
            minq_pi = torch.min(self._q(self.q1, s, an), self._q(self.q2, s, an))
            lpi = (self.alpha.detach() * lp - minq_pi).mean()
            self.opt_pi.zero_grad()
            lpi.backward()
            self.opt_pi.step()
            if self.auto:
                la = -(self.log_alpha * (lp + self.target_entropy).detach()).mean()
                self.opt_alpha.zero_grad()
                la.backward()
                self.opt_alpha.step()
                self.alpha = self.log_alpha.exp()
            with torch.no_grad():
                for tgt, src in ((self.q1t, self.q1), (self.q2t, self.q2)):
                    for t, p in zip(tgt, src):
                        t.copy_(tau * p.data + (1.0 - tau) * t)
            self.last = {"y": y, "q1_loss": l1.detach(), "q2_loss": l2.detach(), "policy_loss": lpi.detach(), "lp": lp.detach(),
                         "q1": q1v.detach(), "q2": q2v.detach()}

    return WeightedPort(obs, act, cfg, capacity=capacity)


def _buf(cap, obs=3, act=2, **kw):
    from sac.replay_buffer import PrioritizedReplayBuffer
    return PrioritizedReplayBuffer(cap, obs, act, device="cuda", **kw)


def _push_dev(buf, n, seed=0):
    s, a, r, s2, d = synth_transitions(n, buf.obs_dim, buf.act_dim, seed)
    t = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32)).cuda()
    for i in range(0, n, buf.capacity):                    # one push_n_dev call stores at most a ring's worth
        k = slice(i, min(n, i + buf.capacity))
        buf.push_device(t(s[k]), t(a[k]), t(r[k]), t(s2[k]), t(d[k]))
    buf.slot_priorities()                 # the tree takes in the pushes: later write-backs name stored transitions


def _sample_u(buf, U, beta=1.0):
    idx, w = buf.sample_with_uniforms(torch.as_tensor(np.asarray(U, dtype=np.float32)), beta)
    return idx.cpu().numpy(), w.cpu().numpy()


def _check_exact_sampling(buf, leaves, rng, B=256, beta=1.0):
    from oracle import per_numpy as P
    pushes = int(buf._lib.sacx_ring_pushes(buf.handle, 0))
    U = rng.random(B).astype(np.float32)
    U[0], U[-1] = 0.0, np.float32(1.0 - 2.0 ** -24)            # edge draws: u = 0 and u -> sum(p)
    idx, w = _sample_u(buf, U, beta)
    slots = P.logical_to_slot(idx, pushes, buf.capacity)
    want = P.sample(leaves, P.strata_u_f32(U, leaves.sum()))
    assert np.array_equal(slots, want)
    assert idx.min() >= 0 and idx.max() < len(buf) and np.all(leaves[slots] > 0)
    ww = P.weights(leaves, leaves[slots], beta)
    assert np.max(np.abs(w - ww) / ww) < 1e-6


@pytest.mark.parametrize("cap,pushes", [(1 << 20, 1 << 20), (5000, 7300)])
def test_tree_write_back_rounds_keep_exact_sums(cap, pushes):
    """Many random write-back rounds (duplicates included) on a full 2^20 ring and on a wrapped 5000-slot ring (not a multiple
    of 32): the leaves equal the sequential oracle, the tree's sampling equals searchsorted over the exact prefix sums, and the
    root min gives weights (p / p_min)^-1."""
    from oracle import per_numpy as P
    buf = _buf(cap, alpha=1.0, eps=0.5)
    _push_dev(buf, pushes)
    rng = np.random.default_rng(1)
    leaves, pmax = buf.slot_priorities()
    leaves = leaves.cpu().numpy().astype(np.float64)
    assert pmax == 1.0 and np.all(leaves == 1.0)                 # every stored transition enters at p_max = 1
    for rnd in range(25):
        B = int(rng.integers(1, 4096))
        _check_exact_sampling(buf, leaves, rng, B=min(B, 1024))   # also records the logical -> slot map of the write-back
        j = rng.integers(0, len(buf), B)
        td = rng.integers(0, 8, B).astype(np.float32) + 0.5       # p = td + 0.5: integers 1..8
        buf.update_priorities(torch.as_tensor(j), torch.as_tensor(td))
        leaves, pmax = P.write_back(leaves, P.logical_to_slot(j, pushes, cap), td.astype(np.float64) + 0.5, pmax)
        got, gmax = buf.slot_priorities()
        assert np.array_equal(got.cpu().numpy(), leaves.astype(np.float32)), rnd
        assert gmax == pmax
    _check_exact_sampling(buf, leaves, rng)


def test_edge_draws_on_a_partly_filled_ring():
    buf = _buf(4096)
    _push_dev(buf, 1000)
    rng = np.random.default_rng(2)
    leaves = np.zeros(4096)
    leaves[:1000] = rng.integers(1, 50, 1000)
    leaves[[0, 1, 999]] = 0.0                                  # zero-priority stored slots are never drawn either
    buf.load_slot_priorities(torch.as_tensor(leaves, dtype=torch.float32), 50.0)
    for _ in range(5):
        _check_exact_sampling(buf, leaves, rng, B=int(rng.integers(1, 700)), beta=float(rng.random()))


def test_philox_draws_follow_the_priorities():
    from scipy.stats import chisquare
    buf = _buf(1000)
    _push_dev(buf, 1000)
    p = 0.995 ** np.arange(1000)
    buf.load_slot_priorities(torch.as_tensor(p, dtype=torch.float32), 1.0)
    idx = torch.empty(256, dtype=torch.int64, device="cuda")
    w = torch.empty(256, dtype=torch.float32, device="cuda")
    counts = torch.zeros(1000, dtype=torch.int64, device="cuda")
    from sac import _engine as E
    for c in range(2000):
        E.check(buf._lib.sacx_per_sample(buf.per_handle, 256, 0.4, None, 1234, c, idx.data_ptr(), w.data_ptr()))
        counts += torch.bincount(idx, minlength=1000)
    counts = counts.cpu().numpy()
    exp = p / p.sum() * counts.sum()
    assert chisquare(counts, exp).pvalue > 1e-3
    # the stream is keyed by (seed, counter): a repeated key repeats the batch, another counter does not
    a = torch.empty_like(idx); b = torch.empty_like(idx)
    E.check(buf._lib.sacx_per_sample(buf.per_handle, 256, 0.4, None, 1234, 5, a.data_ptr(), w.data_ptr()))
    E.check(buf._lib.sacx_per_sample(buf.per_handle, 256, 0.4, None, 1234, 5, b.data_ptr(), w.data_ptr()))
    assert torch.equal(a, b)
    E.check(buf._lib.sacx_per_sample(buf.per_handle, 256, 0.4, None, 1234, 6, b.data_ptr(), w.data_ptr()))
    assert not torch.equal(a, b)


def test_new_pushes_and_wrap_take_p_max():
    buf = _buf(100, alpha=1.0, eps=0.5)
    s, a, r, s2, d = synth_transitions(200, 3, 2, 5)
    buf.push_batch(s[:60], a[:60], r[:60], s2[:60], d[:60].astype(np.float32))      # host staging path
    buf.slot_priorities()
    buf.update_priorities(torch.arange(10), torch.full((10,), 6.5))                     # p = 7 -> p_max = 7
    buf.update_priorities(torch.arange(10, 20), torch.full((10,), 1.5))                 # p = 2
    buf.push_batch(s[60:70], a[60:70], r[60:70], s2[60:70], d[60:70].astype(np.float32))
    leaves, pmax = buf.slot_priorities()
    leaves = leaves.cpu().numpy()
    assert pmax == 7.0
    assert np.all(leaves[:10] == 7.0) and np.all(leaves[10:20] == 2.0) and np.all(leaves[20:60] == 1.0)
    assert np.all(leaves[60:70] == 7.0) and np.all(leaves[70:] == 0.0)
    t = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32)).cuda()
    buf.update_priorities(torch.arange(0, 70), torch.full((70,), 2.5))                  # p = 3 everywhere
    buf.push_device(t(s[70:120]), t(a[70:120]), t(r[70:120]), t(s2[70:120]), t(d[70:120]))   # slots 70..99, then 0..19 (overwritten)
    leaves = buf.slot_priorities()[0].cpu().numpy()
    assert np.all(leaves[70:] == 7.0) and np.all(leaves[:20] == 7.0) and np.all(leaves[20:70] == 3.0)
    assert np.array_equal(buf.priorities().cpu().numpy()[:50], leaves[20:70])          # logical order starts at the oldest slot


def test_duplicate_write_back_highest_row_wins_deterministically():
    runs = []
    for _ in range(2):
        buf = _buf(64, alpha=0.7, eps=1e-3)
        _push_dev(buf, 64)
        rng = np.random.default_rng(9)
        j = torch.as_tensor(np.concatenate([[3, 3, 3, 7], rng.integers(0, 64, 4000)]))
        td = torch.as_tensor(np.concatenate([[1.0, 2.0, 3.0, 4.0], rng.random(4000) * 3]).astype(np.float32))
        buf.update_priorities(j, td)
        leaves = buf.slot_priorities()[0].cpu().numpy()
        last = {}
        for k, s in enumerate(j.tolist()):
            last[s] = k
        want = np.ones(64, np.float32)
        for s, k in last.items():
            want[s] = np.float32((np.float32(td[k]) + np.float32(1e-3)) ** np.float32(0.7))
        assert np.allclose(leaves, want, rtol=1e-6, atol=0)
        runs.append(leaves)
    assert np.array_equal(runs[0], runs[1])


# ---------------------------------------------------------------------------------------------------- the agent's update
PATHS = [("rowpar", {}, 256), ("tiles", {"SACX_ROWPAR": "0", "SACX_TC": "0"}, 256), ("tc", {"SACX_TC_MIN_BATCH": "1024"}, 1024)]


def _agent(monkeypatch, env, batch, prioritized, obs=8, act=2, capacity=3000, seed=0):
    from sac.agent import SAC
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cfg = base_config(hidden=(256, 256), batch=batch, capacity=capacity, rng="device", seed=seed)
    if prioritized is not None:
        cfg["buffer"]["prioritized"] = prioritized
    a = SAC(FakeEnv(obs, act), cfg)
    for k in env:
        monkeypatch.delenv(k)
    return a, cfg


def _fill(agent, n, seed=3):
    s, a, r, s2, d = synth_transitions(n, agent.obs_size, agent.action_size, seed)
    agent.replay_buffer.push_batch(s, a, r, s2, d.astype(np.float32))
    return s, a, r, s2, d.astype(np.float32)


def _path_of(agent):
    eng = agent.engine
    return "tc" if eng.tensor_core()[0] else eng.path()[0]


VIEWS = ("block.params", "block.targets", "block.m", "block.v", "out.y", "out.q1", "out.q2", "out.logpi", "scal.log_alpha")


@pytest.mark.parametrize("name,env,batch", PATHS)
def test_unit_weights_are_bit_identical_to_the_uniform_update(monkeypatch, name, env, batch):
    """beta = 0: every weight is exactly 1, and a PER update equals sacx_update without PER given the same indices and eps."""
    a, _ = _agent(monkeypatch, env, batch, {"alpha": 0.6, "beta": 0.0})
    u, _ = _agent(monkeypatch, env, batch, None)
    assert _path_of(a) == _path_of(u) == name
    _fill(a, 3000); _fill(u, 3000)
    u.engine.arena.copy_(a.engine.arena)
    torch.manual_seed(0)
    for step in range(3):
        e1 = torch.randn(batch, 2, device="cuda"); e2 = torch.randn(batch, 2, device="cuda")
        a.engine.update(None, e1, e2, 1)
        idx = a.engine.view("batch.idx").clone().reshape(-1)
        u.engine.update(idx, e1, e2, 1)
        torch.cuda.synchronize()
        for v in VIEWS:
            assert torch.equal(a.engine.view(v), u.engine.view(v)), (name, step, v)
        ma, mu = a.engine.metrics(), u.engine.metrics()
        assert ma == mu, (name, step)


@pytest.mark.parametrize("name,env,batch", PATHS)
def test_weighted_update_matches_the_torch_port(monkeypatch, name, env, batch):
    """beta = 1 with spread priorities: one update against the torch port with the weighted critic loss from the same state;
    afterwards the sampled slots hold (delta + eps)^alpha of the update's own q1 / q2 / y."""
    from oracle import per_numpy as P
    per = {"alpha": 0.6, "beta": 1.0, "eps": 1e-6}
    a, cfg = _agent(monkeypatch, env, batch, per)
    assert _path_of(a) == name
    S, A, R, S2, D = _fill(a, 3000)
    rng = np.random.default_rng(4)
    p = rng.uniform(0.05, 5.0, 3000)
    a.replay_buffer.load_slot_priorities(torch.as_tensor(p, dtype=torch.float32), 5.0)
    p = p.astype(np.float32).astype(np.float64)
    port = _weighted_port(a.obs_size, a.action_size, cfg, capacity=3000)
    eng = a.engine
    for tag, dst in (("pi", port.pi), ("q1", port.q1), ("q2", port.q2), ("q1t", port.q1t), ("q2t", port.q2t)):
        for l in range(len(dst) // 2):
            dst[2 * l].data.copy_(eng.view(f"{tag}.W{l}").cpu())
            dst[2 * l + 1].data.copy_(eng.view(f"{tag}.b{l}").cpu().reshape(dst[2 * l + 1].shape))
    torch.manual_seed(1)
    e1 = torch.randn(batch, 2, device="cuda"); e2 = torch.randn(batch, 2, device="cuda")
    eng.update(None, e1, e2, 1)
    torch.cuda.synchronize()
    idx = eng.view("batch.idx").cpu().numpy().reshape(-1)
    w = P.weights(p, p[idx], 1.0)                                   # ring never wrapped: slot = logical index
    assert w.max() <= 1.0
    t = lambda x: torch.as_tensor(x)
    port.update_from_batch(t(S[idx]), t(A[idx]), t(R[idx]), t(S2[idx]), t(D[idx]), e1.cpu(), e2.cpu(), w)
    ref = port.last
    assert rel_l2(eng.view("out.y").cpu().numpy().ravel(), ref["y"].numpy().ravel()) < 2e-5
    assert rel_l2(eng.view("out.q1").cpu().numpy().ravel(), ref["q1"].numpy().ravel()) < 2e-5
    assert rel_l2(eng.view("out.logpi").cpu().numpy().ravel(), ref["lp"].numpy().ravel()) < 2e-5
    m = eng.metrics()
    assert abs(m["q1_loss"] - float(ref["q1_loss"])) <= 2e-5 * abs(float(ref["q1_loss"])) + 1e-7
    for tag, src in (("q1", port.q1), ("q2", port.q2), ("pi", port.pi)):
        for l in range(len(src) // 2):
            assert rel_l2(eng.view(f"{tag}.W{l}").cpu().numpy(), src[2 * l].detach().numpy()) < 3e-4, (name, tag, l)
    # priority refresh (applied by the read)
    q1, q2, y = (eng.view(v).cpu().numpy().ravel() for v in ("out.q1", "out.q2", "out.y"))
    leaves = a.replay_buffer.slot_priorities()[0].cpu().numpy()
    want = P.priority(P.td_delta(q1, q2, y), 0.6, 1e-6)
    last = {}
    for k, s in enumerate(idx.tolist()):
        last[s] = k
    got = np.array([leaves[s] for s in last]); exp = np.array([want[k] for k in last.values()])
    assert np.max(np.abs(got - exp) / exp) < 1e-5


def test_burst_equals_single_steps_with_the_beta_schedule(monkeypatch):
    per = {"alpha": 0.6, "beta": 0.4, "beta_steps": 6}
    a, _ = _agent(monkeypatch, {}, 256, per)
    b, _ = _agent(monkeypatch, {}, 256, per)
    _fill(a, 2000); _fill(b, 2000)
    a.training_steps(10)
    for _ in range(10):
        b.training_step()
    torch.cuda.synchronize()
    for v in VIEWS + ("batch.idx",):
        assert torch.equal(a.engine.view(v), b.engine.view(v)), v
    la, pa = a.replay_buffer.slot_priorities()
    lb, pb = b.replay_buffer.slot_priorities()
    assert torch.equal(la, lb) and pa == pb
    assert int(a.engine.view("scal.updates")) == 10


def test_snapshot_resumes_bit_exactly(monkeypatch, tmp_path):
    import random
    per = {"alpha": 0.6, "beta": 0.4, "beta_steps": 20}
    from sac.agent import SAC
    cfg = base_config(hidden=(64, 64), batch=64, capacity=500, rng="device")
    cfg["buffer"]["prioritized"] = per
    a = SAC(FakeEnv(6, 2), cfg)
    s, ac, r, s2, d = synth_transitions(700, 6, 2, 4)
    for i in range(700):
        a.store_transition(s[i], ac[i], float(r[i]), s2[i], bool(d[i]))
    random.seed(3); torch.manual_seed(3)
    for _ in range(5):
        a.training_step()
    path = str(tmp_path / "snap.pt")
    a.save_snapshot(path)
    for i in range(3):
        a.store_transition(s[i], ac[i], 0.5, s2[i], False)
        a.training_step()
    b = SAC(FakeEnv(6, 2), cfg)
    for i in range(80):
        b.store_transition(s[i] * 3, ac[i], 1.0, s2[i], False)
    b.training_step()
    b.load_snapshot(path)
    for i in range(3):
        b.store_transition(s[i], ac[i], 0.5, s2[i], False)
        b.training_step()
    for n in ("block.params", "block.targets", "block.m", "block.v", "batch.idx"):
        assert torch.equal(a.engine.view(n), b.engine.view(n)), n
    la, pa = a.replay_buffer.slot_priorities()
    lb, pb = b.replay_buffer.slot_priorities()
    assert torch.equal(la, lb) and pa == pb
    # a snapshot without priorities cannot resume a prioritized agent
    u = SAC(FakeEnv(6, 2), base_config(hidden=(64, 64), batch=64, capacity=500, rng="device"))
    for i in range(100):
        u.store_transition(s[i], ac[i], float(r[i]), s2[i], bool(d[i]))
    u.save_snapshot(str(tmp_path / "uniform.pt"))
    with pytest.raises(ValueError):
        SAC(FakeEnv(6, 2), cfg).load_snapshot(str(tmp_path / "uniform.pt"))


def test_refusals(monkeypatch):
    from sac.agent import SAC
    from sac.population import DataParallelSAC, SACPopulation
    cfg = base_config(hidden=(64, 64), batch=64, capacity=500, rng="host")
    cfg["buffer"]["prioritized"] = {"alpha": 0.6}
    with pytest.raises(ValueError):
        SAC(FakeEnv(6, 2), cfg)
    cfg["train"]["rng"] = "device"
    with pytest.raises(ValueError):
        SACPopulation(6, 2, cfg, n_agents=2)
    with pytest.raises(ValueError):
        DataParallelSAC(6, 2, cfg, global_batch=64)
    a = SAC(FakeEnv(6, 2), cfg)
    _fill(a, 200)
    with pytest.raises(ValueError):
        a.engine.update(torch.arange(64, device="cuda"), None, None, 1)
    with pytest.raises(ValueError):
        a.engine.update_host(np.arange(64), None, None, 1)
    with pytest.raises(ValueError):
        a.engine.update(None, None, None, 1, staged=True)
    a.training_step()                                              # the refused calls left the agent usable
    assert int(a.engine.view("scal.updates")) == 1


def test_main_process_learns_point_mass_with_prioritized_replay(tmp_path):
    import yaml
    cfg = base_config(hidden=(256, 256), batch=256, auto=False, alpha=0.02, rng="device")
    cfg["train"].update(warming_steps=1000, num_episodes=400, device="cuda")
    cfg["logger"].update(env_name="OneDPointMassReachEnv", enabled=False)
    cfg["buffer"]["prioritized"] = {"alpha": 0.6, "beta": 0.4, "beta_steps": 20000, "eps": 1e-6}
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
    assert final >= 0.80, f"last-100 average return {final} with prioritized replay"
