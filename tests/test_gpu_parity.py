"""-m gpu parity tests: the CUDA path (through the C ABI / the `sac` binding) against the oracle and the
golden vectors recorded from the real reference.

Tolerances (SURVEY section 8c): indices and gathered batches bit-exact; teacher-forced single updates
y / logpi / q rel-L2 <= 2e-5, gradients <= 5e-5, parameters / Adam moments <= 1e-4 (Adam's first steps are
lr*sign(g), so noise-level gradient elements may flip: norm-relative metric), log_alpha abs <= 1e-6.
"""
import json
import os
import random

import numpy as np
import pytest
import torch

from gpu_helpers import FakeEnv, assert_close, base_config, dev, engine_from_golden, fill_ring, load_nets, read_net
from helpers import Golden, numpy_oracle_from_golden, rel_l2, synth_transitions

pytestmark = pytest.mark.gpu

SMALL = ["tiny_auto", "tiny_fixed", "outact_tanh"] + [f"acts_{a}" for a in
                                                      ("relu", "tanh", "elu", "leaky_relu", "gelu", "selu", "identity")]


# ----------------------------------------------------------------------------- ring (a1-a3)
def test_ring_gather_bit_exact_vs_reference_stream(golden_dir):
    """Indices: Python's own random.sample stream; gathered rows must equal what the reference returned."""
    from sac.replay_buffer import ReplayBuffer

    with open(os.path.join(golden_dir, "sampling.json")) as f:
        g = json.load(f)
    for c in g["cases"]:
        n, k, cap = c["pushes"], c["k"], c["capacity"]
        rb = ReplayBuffer(cap, 3, 2)
        ids = np.arange(n, dtype=np.float32)
        s = np.stack([ids, ids + 0.25, -ids], 1)
        a = np.stack([ids, ids * 2], 1)
        rb.push_batch(s, a, ids, s + 1, (np.arange(n) % 7 == 0).astype(np.float32))
        assert len(rb) == min(n, cap)
        random.seed(c["seed"])
        for want in c["push_ids"]:
            batch = rb.sample_tensors(k)                      # draws random.sample(range(len), k) like the reference
            got = batch.reward.cpu().numpy()
            assert np.array_equal(got, np.asarray(want, dtype=np.float32))
            w = np.asarray(want)
            assert np.array_equal(batch.state.cpu().numpy(), s[w])
            assert np.array_equal(batch.action.cpu().numpy(), a[w])
            assert np.array_equal(batch.next_state.cpu().numpy(), s[w] + 1)
            assert np.array_equal(batch.done.cpu().numpy(), (w % 7 == 0).astype(np.float32))


def test_ring_single_push_wrap_and_legacy_sample():
    from sac.replay_buffer import ReplayBuffer, Transition

    rb = ReplayBuffer(50)
    with pytest.raises(ValueError):
        rb._require(1)
    for p in range(120):                                        # wraps 2.4x, one push at a time (lazy allocation)
        rb.push(np.full(4, p, np.float64), [p, -p], float(p), np.full(4, p + 0.5), p % 3 == 0)
    assert len(rb) == 50 and len(rb.memory) == 50
    with pytest.raises(ValueError, match="Not enough samples"):
        rb.sample(51)
    random.seed(3)
    rows = rb.sample(20)
    random.seed(3)
    logical = random.sample(range(50), 20)
    assert isinstance(rows[0], Transition)
    assert [int(t.reward) for t in rows] == [70 + j for j in logical]      # oldest survivor is push 70
    assert all(t.done == (int(t.reward) % 3 == 0) for t in rows)
    assert rows[0].state.dtype == np.float32 and rows[0].state.shape == (4,)


def test_device_index_sampler_is_without_replacement():
    from sac.replay_buffer import ReplayBuffer

    rb = ReplayBuffer(100000, 2, 1)
    n = 70000
    z = np.zeros((n, 2), np.float32)
    rb.push_batch(z, z[:, :1], np.arange(n), z, np.zeros(n))
    counts = np.zeros(n)
    for c in range(50):
        idx = rb.device_indices(1024, seed=7, counter=c).cpu().numpy()
        assert idx.min() >= 0 and idx.max() < n and len(np.unique(idx)) == 1024
        counts[idx] += 1
    # roughly uniform: mean index near n/2; occupancy follows Poisson(lambda = 51200/70000)
    hit = np.nonzero(counts)[0]
    lam = 50 * 1024 / n
    assert abs(hit.mean() / n - 0.5) < 0.02 and counts.max() <= 10
    assert abs(len(hit) / n - (1 - np.exp(-lam))) < 0.01
    # tiny populations, including k == n
    rb2 = ReplayBuffer(16, 2, 1)
    rb2.push_batch(z[:12], z[:12, :1], np.arange(12), z[:12], np.zeros(12))
    assert sorted(rb2.device_indices(12, 1, 0).cpu().numpy().tolist()) == list(range(12))


# ----------------------------------------------------------------------------- staged phases (a5-a11)
def _flat(dW, db):
    out = {}
    for l, (w, b) in enumerate(zip(dW, db)):
        out[f"net.{2 * l}.weight"] = w
        out[f"net.{2 * l}.bias"] = b
    return out


@pytest.mark.parametrize("name", SMALL)
def test_staged_update_teacher_forced(name):
    """Each reference method's CUDA counterpart against the golden (= reference) values, per update, starting
    from the reference's recorded state."""
    g = Golden(name)
    eng = engine_from_golden(g)
    o = numpy_oracle_from_golden(g)
    S, A, R, S2, D = synth_transitions(g.n_fill, g.obs, g.act)
    D = D.astype(np.float32)
    nl_pi, nl_q = len(g.cfg["policy_net"]["hidden_sizes"]) + 1, len(g.cfg["q_net"]["hidden_sizes"]) + 1
    auto = g.cfg["sac"]["auto_entropy_tuning"]
    for k in range(g.K):
        idx = g[f"step{k}/idx"]
        s, a, r, s2, d = S[idx], A[idx], R[idx], S2[idx], D[idx]
        e1, e2 = g[f"step{k}/eps1"], g[f"step{k}/eps2"]
        eng.load_batch(dev(s), dev(a), dev(r), dev(s2), dev(d))
        # a6 target
        y = torch.empty(len(idx), device="cuda")
        eng.target(dev(e1), y)
        assert_close("y", y.cpu().numpy(), g[f"step{k}/y"], 2e-5)
        # a7 critic gradients, then the step
        eng.critic_step(y, grads_only=True)
        for tag, key in (("q1", "gq1"), ("q2", "gq2")):
            ref = g.sd(f"step{k}/{key}")
            got = read_net(eng, tag, nl_q, prefix="g.")
            for nm in ref:
                assert_close(f"grad {tag}.{nm}", got[nm], ref[nm], 5e-5)
        assert_close("q1", eng.view("out.q1").cpu().numpy().ravel(), g[f"step{k}/q1"], 2e-5)
        eng.critic_step(dev(g[f"step{k}/y"]))
        m = eng.metrics()
        assert abs(m["q1_loss"] - float(g[f"step{k}/q1_loss"])) <= 2e-5 * abs(float(g[f"step{k}/q1_loss"])) + 1e-7
        assert abs(m["q2_loss"] - float(g[f"step{k}/q2_loss"])) <= 2e-5 * abs(float(g[f"step{k}/q2_loss"])) + 1e-7
        for tag in ("q1", "q2"):
            ref = g.sd(f"step{k}/{tag}")
            got = read_net(eng, tag, nl_q)
            for nm in ref:
                assert_close(f"param {tag}.{nm}", got[nm], ref[nm], 1e-4)
        # teacher-force the critics to the reference's post-step values before the actor phase
        load_nets(eng, {"q1": g.sd(f"step{k}/q1"), "q2": g.sd(f"step{k}/q2")})
        # a8 actor gradients, then the step
        lp = torch.empty(len(idx), device="cuda")
        eng.actor_step(dev(e2), lp, grads_only=True)
        assert_close("logpi", lp.cpu().numpy(), g[f"step{k}/lp"], 2e-5)
        ref = g.sd(f"step{k}/gpi")
        got = read_net(eng, "pi", nl_pi, prefix="g.")
        for nm in ref:
            assert_close(f"grad pi.{nm}", got[nm], ref[nm], 5e-5)
        eng.actor_step(dev(e2), lp)
        ref = g.sd(f"step{k}/pi")
        got = read_net(eng, "pi", nl_pi)
        for nm in ref:
            assert_close(f"param pi.{nm}", got[nm], ref[nm], 1e-4)
        # a9 temperature
        if auto:
            info = eng.alpha_step(dev(g[f"step{k}/lp"]), want_metrics=True)
            la = float(eng.view("scal.log_alpha").item())
            assert abs(la - float(g[f"step{k}/log_alpha"])) < 1e-6
            assert abs(info["alpha"] - float(g[f"step{k}/alpha"])) < 1e-6
            assert abs(info["alpha_loss"] - float(g[f"step{k}/alpha_loss"])) < 2e-5 * max(1.0, abs(float(g[f"step{k}/alpha_loss"])))
        # a10 Polyak: bit-exact given identical inputs (separately rounded products)
        load_nets(eng, {"q1": g.sd(f"step{k}/q1"), "q2": g.sd(f"step{k}/q2")})
        if k > 0:
            load_nets(eng, {"q1t": g.sd(f"step{k - 1}/q1t"), "q2t": g.sd(f"step{k - 1}/q2t")})
        else:
            load_nets(eng, {"q1t": g.sd("init/q1"), "q2t": g.sd("init/q2")})
        eng.polyak()
        for tag in ("q1t", "q2t"):
            ref = g.sd(f"step{k}/{tag}")
            got = read_net(eng, tag, nl_q)
            for nm in ref:
                assert np.array_equal(got[nm], ref[nm]), f"polyak {tag}.{nm}"
        # continue from the reference's exact state (policy too)
        load_nets(eng, {"pi": g.sd(f"step{k}/pi")})


@pytest.mark.parametrize("name", SMALL + ["bipedal", "pendulum128"])
def test_fused_update_free_running_vs_reference(name):
    """K consecutive fused updates (ring gather included) from the reference's initial weights with the
    reference's recorded index stream and normals; compared with the reference's own outputs."""
    from sac.replay_buffer import ReplayBuffer

    g = Golden(name)
    eng = engine_from_golden(g)
    rb = ReplayBuffer(g.cfg["buffer"]["capacity"], g.obs, g.act)
    fill_ring(rb, g.n_fill, g.obs, g.act)
    eng.attach_ring(rb)
    nl_pi, nl_q = len(g.cfg["policy_net"]["hidden_sizes"]) + 1, len(g.cfg["q_net"]["hidden_sizes"]) + 1
    auto = g.cfg["sac"]["auto_entropy_tuning"]
    for k in range(g.K):
        m = eng.update_host(g[f"step{k}/idx"], g[f"step{k}/eps1"], g[f"step{k}/eps2"], 1)
        tol = 3e-5 * (3 ** k)             # chaotic growth of fp32 differences over free-running steps (F16)
        assert_close(f"step{k} y", eng.view("out.y").cpu().numpy().ravel(), g[f"step{k}/y"], tol)
        assert_close(f"step{k} logpi", eng.view("out.logpi").cpu().numpy().ravel(), g[f"step{k}/lp"], tol)
        assert abs(m["q1_loss"] - float(g[f"step{k}/q1_loss"])) <= 10 * tol * abs(float(g[f"step{k}/q1_loss"])) + 1e-7
        assert m["nonfinite"] == 0 and m["updates"] == k + 1
        if auto:
            assert abs(m["log_alpha"] - float(g[f"step{k}/log_alpha"])) < 2e-6
        for tag, nl in (("pi", nl_pi), ("q1", nl_q), ("q2", nl_q), ("q1t", nl_q), ("q2t", nl_q)):
            got = read_net(eng, tag, nl)
            for nm, v in got.items():
                key = f"step{k}/{tag}/{nm}"
                if g.full:
                    assert_close(key, v, g[key], 1e-4 * (2 ** k))
                else:
                    assert_close(key + "#smp", v.ravel()[::97], g[key + "#smp"], 1e-4 * (2 ** k))
                    v64 = v.astype(np.float64).ravel()
                    assert abs((v64 * v64).sum() - g[key + "#chk"][1]) <= 1e-4 * g[key + "#chk"][1] + 1e-12


def test_fused_equals_per_phase_launches(monkeypatch):
    """The persistent cooperative tile-parallel kernel and one-launch-per-phase execute the same op table: identical
    bits. (SACX_ROWPAR=0: the row-parallel kernel is a different summation order, compared in test_gpu_rowpar.py.)"""
    from sac.replay_buffer import ReplayBuffer

    monkeypatch.setenv("SACX_ROWPAR", "0")
    g = Golden("bipedal")
    res = []
    for staged in (False, True):
        eng = engine_from_golden(g)
        rb = ReplayBuffer(g.cfg["buffer"]["capacity"], g.obs, g.act)
        fill_ring(rb, g.n_fill, g.obs, g.act)
        eng.attach_ring(rb)
        idx = torch.stack([dev(g[f"step{k}/idx"]) for k in range(g.K)])
        e1 = torch.stack([dev(g[f"step{k}/eps1"]) for k in range(g.K)])
        e2 = torch.stack([dev(g[f"step{k}/eps2"]) for k in range(g.K)])
        eng.update(idx, e1, e2, n_steps=g.K, staged=staged)          # K steps inside one launch vs 17*K launches
        eng.sync()
        res.append(eng.view("block.params").cpu().numpy().copy())
        assert eng.metrics()["updates"] == g.K
    assert np.array_equal(res[0], res[1])


def test_device_rng_mode_update_matches_oracle():
    """Throughput mode: indices and normals generated in-kernel. Read them back and replay the oracle."""
    from sac.replay_buffer import ReplayBuffer

    g = Golden("acts_elu")
    eng = engine_from_golden(g)
    rb = ReplayBuffer(200, g.obs, g.act)
    S, A, R, S2, D = fill_ring(rb, 150, g.obs, g.act)
    eng.attach_ring(rb)
    o = numpy_oracle_from_golden(g)
    B = g.cfg["train"]["batch_size"]
    seen = []
    for k in range(3):
        eng.update(None, None, None, 1)
        eng.sync()
        idx = eng.view("batch.idx").cpu().numpy().ravel()
        e1 = eng.view("batch.eps1").cpu().numpy()
        e2 = eng.view("batch.eps2").cpu().numpy()
        assert len(np.unique(idx)) == B and idx.min() >= 0 and idx.max() < 150
        seen.append(e1.copy())
        o.update(S[idx], A[idx], R[idx], S2[idx], D[idx], e1, e2)
        assert_close("y", eng.view("out.y").cpu().numpy().ravel(), o.last["y"], 1e-4)
        assert_close("logpi", eng.view("out.logpi").cpu().numpy().ravel(), o.last["lp"], 1e-4)
        assert abs(float(eng.view("scal.log_alpha").item()) - float(o.log_alpha)) < 5e-6
    assert not np.array_equal(seen[0], seen[1])                     # counter advances the streams
    allz = np.concatenate([s.ravel() for s in seen])
    assert abs(allz.mean()) < 0.35 and 0.6 < allz.std() < 1.4


def test_device_normals_are_standard():
    from sac.replay_buffer import ReplayBuffer

    cfg = base_config(hidden=(32, 32), batch=4096, rng="device")
    from sac.engine import UpdateEngine
    eng = UpdateEngine(6, 4, cfg)
    for tag, nl in (("pi", 3), ("q1", 3), ("q2", 3)):
        for l in range(nl):
            eng.view(f"{tag}.W{l}").normal_(0, 0.1)
    eng.reset_state()
    rb = ReplayBuffer(10000, 6, 4)
    fill_ring(rb, 8000, 6, 4)
    eng.attach_ring(rb)
    eng.update(None, None, None, 1)
    z = torch.cat([eng.view("batch.eps1").reshape(-1), eng.view("batch.eps2").reshape(-1)]).cpu().numpy()
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02
    assert abs((z ** 3).mean()) < 0.06 and abs((z ** 4).mean() - 3) < 0.15
    assert abs(np.corrcoef(z[:-1], z[1:])[0, 1]) < 0.02


# ----------------------------------------------------------------------------- population (8e) on one GPU
def test_population_agents_are_independent_and_match_single_agent():
    from sac.engine import UpdateEngine
    from sac.replay_buffer import ReplayBuffer

    g = Golden("acts_tanh")
    n_agents = 5
    pop = UpdateEngine(g.obs, g.act, g.cfg, n_agents=n_agents)
    ring = ReplayBuffer(100, g.obs, g.act, n_agents=n_agents)
    B, K = g.cfg["train"]["batch_size"], 2
    rng = np.random.default_rng(5)
    idx = rng.integers(0, 64, (K, n_agents, B)).astype(np.int64)
    e1 = rng.standard_normal((K, n_agents, B, g.act)).astype(np.float32)
    e2 = rng.standard_normal((K, n_agents, B, g.act)).astype(np.float32)
    singles = []
    for ag in range(n_agents):
        sds = {t: {k: (v * (1 + 0.1 * ag)).astype(np.float32) for k, v in g.sd(f"init/{t}").items()} for t in ("pi", "q1", "q2")}
        load_nets(pop, sds, agent=ag)
        fill_ring(ring, 64, g.obs, g.act, seed=ag, agent=ag)
        one = UpdateEngine(g.obs, g.act, g.cfg)
        load_nets(one, sds)
        one.reset_state()
        r1 = ReplayBuffer(100, g.obs, g.act)
        fill_ring(r1, 64, g.obs, g.act, seed=ag)
        one.attach_ring(r1)
        one.update(dev(idx[:, ag]), dev(e1[:, ag]), dev(e2[:, ag]), n_steps=K)
        one.sync()
        singles.append(one.view("block.params").cpu().numpy().copy())
    pop.reset_state()
    pop.attach_ring(ring)
    pop.update(dev(idx), dev(e1), dev(e2), n_steps=K)
    pop.sync()
    for ag in range(n_agents):
        got = pop.view("block.params", ag).cpu().numpy()
        # different tile configuration (64x64 vs 32x32) => different summation order: tolerance, not bits
        assert_close(f"agent {ag} params", got, singles[ag], 2e-5)
        assert pop.metrics(ag)["updates"] == K


# ----------------------------------------------------------------------------- edge shapes
def _random_nets(obs, act, hidden_pi, hidden_q, seed=0, scale=0.3):
    rng = np.random.default_rng(seed)
    sds = {}
    for tag, dims in (("pi", [obs] + list(hidden_pi) + [2 * act]), ("q1", [obs + act] + list(hidden_q) + [1]),
                      ("q2", [obs + act] + list(hidden_q) + [1])):
        sd = {}
        for l in range(len(dims) - 1):
            sd[f"net.{2 * l}.weight"] = (rng.standard_normal((dims[l + 1], dims[l])) * scale).astype(np.float32)
            sd[f"net.{2 * l}.bias"] = (rng.standard_normal(dims[l + 1]) * 0.1).astype(np.float32)
        sds[tag] = sd
    return sds


@pytest.mark.parametrize("obs,act,hp,hq,B,actfn", [
    (7, 5, (33, 17), (19, 23), 50, "tanh"),          # nothing aligned: scalar loaders / epilogues, ragged tiles, B % 8 != 0
    (3, 1, (5,), (6,), 9, "gelu"),                   # single hidden layer, tiny
    (11, 32, (64, 40), (48, 36), 70, "relu"),        # maximum action dimension
    (24, 4, (320, 300), (288, 260), 96, "elu"),      # hidden wider than one 256-wide K ring / register-resident row path
    (6, 2, (16, 16, 16, 16), (12, 12, 12), 40, "selu"),   # deep networks
])
def test_update_edge_shapes_vs_oracle(obs, act, hp, hq, B, actfn):
    """One fused update on awkward shapes against the NumPy oracle (no golden needed: the oracle is pinned)."""
    from oracle.sac_numpy import Hyper, SACOracle, mlp_from_state_dict
    from sac.engine import UpdateEngine
    from sac.replay_buffer import ReplayBuffer
    cfg = base_config(hidden=hp, q_hidden=hq, act=actfn, batch=B, capacity=500)
    eng = UpdateEngine(obs, act, cfg)
    sds = _random_nets(obs, act, hp, hq)
    load_nets(eng, sds)
    eng.reset_state()
    rb = ReplayBuffer(500, obs, act)
    S, A, R, S2, D = fill_ring(rb, 300, obs, act)
    eng.attach_ring(rb)
    o = SACOracle(mlp_from_state_dict(sds["pi"], actfn, "identity"), mlp_from_state_dict(sds["q1"], actfn, "identity"),
                  mlp_from_state_dict(sds["q2"], actfn, "identity"), Hyper())
    rng = np.random.default_rng(3)
    for k in range(2):
        idx = rng.choice(300, B, replace=False).astype(np.int64)
        e1 = rng.standard_normal((B, act)).astype(np.float32)
        e2 = rng.standard_normal((B, act)).astype(np.float32)
        m = eng.update_host(idx, e1, e2, 1)
        o.update(S[idx], A[idx], R[idx], S2[idx], D[idx], e1, e2)
        assert m["nonfinite"] == 0
        assert_close("y", eng.view("out.y").cpu().numpy().ravel(), o.last["y"], 1e-4)
        assert_close("logpi", eng.view("out.logpi").cpu().numpy().ravel(), o.last["lp"], 1e-4)
        assert abs(float(eng.view("scal.log_alpha").item()) - float(o.log_alpha)) < 5e-6
    for tag, net in (("pi", o.pi), ("q1", o.q1), ("q2", o.q2), ("q1t", o.q1t)):
        for l, (w, b) in enumerate(zip(net.W, net.b)):
            assert_close(f"{tag}.W{l}", eng.view(f"{tag}.W{l}").cpu().numpy(), w, 3e-4)
            assert_close(f"{tag}.b{l}", eng.view(f"{tag}.b{l}").cpu().numpy().ravel(), b, 3e-4)


def test_full_size_ring_properties():
    """BASELINE config 2 size: 1M transitions (216 MB). Size-independent properties: the gather of every logical index
    returns the row that was pushed there (round trip, bit-exact) before and after wrap-around."""
    from sac.replay_buffer import ReplayBuffer
    N, O, A = 1_000_000, 24, 4
    rb = ReplayBuffer(N, O, A)
    ids = torch.arange(N + 300_000, device="cuda", dtype=torch.float32)
    for lo in range(0, N + 300_000, 260_000):                 # 1.3M pushes: wraps past capacity
        blk = ids[lo: lo + 260_000]
        s = blk[:, None] + torch.arange(O, device="cuda", dtype=torch.float32)[None, :] * 0.5
        rb.push_device(s, blk[:, None].repeat(1, A), -blk, s + 1, (blk % 2))
    assert len(rb) == N
    oldest = 300_000
    idx = torch.randint(0, N, (65536,), device="cuda")
    got = rb.sample_tensors(65536, indices=idx)
    want = (idx + oldest).float()
    assert torch.equal(got.reward, -want) and torch.equal(got.action[:, 0], want)
    assert torch.equal(got.state[:, 3], want + 1.5) and torch.equal(got.next_state[:, 0], want + 1.0)
    assert torch.equal(got.done, want % 2)
    dev_idx = rb.device_indices(4096, seed=1, counter=9)
    assert dev_idx.unique().numel() == 4096 and int(dev_idx.max()) < N
