"""Pin the two oracles against vectors recorded from the real reference.

* torch_port: same torch ops in the same order => BIT-EXACT (y, logpi, losses, params, log_alpha).
* sac_numpy (hand-derived gradients, numpy matmul): fp32 tolerance -- teacher-forced single
  updates: rel-L2 <= 1e-5 on y/logpi/grads/params; |log_alpha| abs <= 1e-6 (SURVEY section 8c).
"""
import random

import numpy as np
import pytest
import torch

from helpers import Golden, numpy_oracle_from_golden, rel_l2, synth_transitions

SMALL = ["tiny_auto", "tiny_fixed", "outact_tanh"] + [f"acts_{a}" for a in
                                                      ("relu", "tanh", "elu", "leaky_relu", "gelu", "selu", "identity")]
LARGE = ["bipedal", "pendulum128"]
# round 2: BASELINE configs 3 / 4 / 5 themselves, K = 10, runs continued from reference-written checkpoints
ROUND2 = ["cfg3_pendulum256", "cfg4_donkey", "cfg4_donkey_elu", "cfg4_donkey_obs216", "cfg5_b2048", "cfg5_b65536", "bipedal_k10",
          "ckpt_tiny_auto", "ckpt_pendulum128"]
# The golden files were recorded with torch on 8 CPU threads. torch's reductions and MKL's GEMMs split their work by the
# thread count, so the same ops give the same bits only at the same count (12 threads, or 1, already differ in the last bit).
RECORDING_THREADS = 8


@pytest.fixture(autouse=True)
def recording_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(RECORDING_THREADS)
    yield
    torch.set_num_threads(n)


def _port_from_golden(g):
    from oracle.torch_port import TorchPortSAC

    port = TorchPortSAC(g.obs, g.act, g.cfg, capacity=g.cfg["buffer"]["capacity"])
    if g.start_ckpt:
        port.load_checkpoint(torch.load(g.ckpt_path(), map_location="cpu", weights_only=False))
    s, a, r, s2, d = synth_transitions(g.n_fill, g.obs, g.act)
    for i in range(g.n_fill):
        port.push(s[i], a[i], float(r[i]), s2[i], bool(d[i]))
    return port


@pytest.mark.parametrize("name", SMALL + LARGE + ROUND2)
def test_torch_port_bit_exact(name):
    g = Golden(name)
    port = _port_from_golden(g)
    # init recipe (F10) reproduces the reference's starting weights bit for bit
    for tag, ps in (("pi", port.pi), ("q1", port.q1), ("q2", port.q2)):
        sd = g.init_sd(tag)
        for l in range(len(ps) // 2):
            assert np.array_equal(ps[2 * l].detach().numpy(), sd[f"net.{2 * l}.weight"])
            assert np.array_equal(ps[2 * l + 1].detach().numpy(), sd[f"net.{2 * l}.bias"])
    for k in range(g.K):
        info = port.training_step()          # free-running: consumes random + torch RNG like the reference
        for key, mine in (("y", port.last["y"].numpy()), ("lp", port.last["lp"].numpy())):
            ref, sel = g.rows(k, key)
            assert np.array_equal(mine[sel], ref), key
            if g.big:
                v64 = mine.astype(np.float64)
                assert np.array_equal(np.array([v64.sum(), (v64 * v64).sum()]), g[f"step{k}/{key}#chk"]), key
        assert np.array_equal(port.last["q1_loss"].numpy(), g[f"step{k}/q1_loss"])
        assert np.array_equal(port.last["q2_loss"].numpy(), g[f"step{k}/q2_loss"])
        if g.cfg["sac"]["auto_entropy_tuning"]:
            assert info["alpha"] == float(g[f"step{k}/alpha"])
            assert info["alpha_loss"] == float(g[f"step{k}/alpha_loss"])
            assert np.array_equal(port.log_alpha.detach().numpy(), g[f"step{k}/log_alpha"])
        st = port.flat_state()
        for tag in ("pi", "q1", "q2", "q1t", "q2t"):
            n = len(getattr(port, tag)) // 2
            for l in range(n):
                for j, kind in ((2 * l, "weight"), (2 * l + 1, "bias")):
                    key = f"step{k}/{tag}/net.{2 * l}.{kind}"
                    v = st[f"{tag}.{j}"]
                    if g.full:
                        assert np.array_equal(v, g[key]), key
                    else:
                        v64 = v.astype(np.float64).ravel()
                        assert np.array_equal(np.array([v64.sum(), (v64 * v64).sum()]), g[key + "#chk"]), key
                        assert np.array_equal(v.ravel()[::97], g[key + "#smp"]), key


def _flat_grads(dW, db):
    out = {}
    for l, (w, b) in enumerate(zip(dW, db)):
        out[f"net.{2 * l}.weight"] = w
        out[f"net.{2 * l}.bias"] = b
    return out


@pytest.mark.parametrize("name", SMALL)
def test_numpy_oracle_teacher_forced(name):
    """Each update starts from the reference's recorded state (teacher forcing), inputs = recorded idx/eps."""
    from oracle.sac_numpy import mlp_from_state_dict, mlp_to_state_dict

    g = Golden(name)
    o = numpy_oracle_from_golden(g)
    s, a, r, s2, d = synth_transitions(g.n_fill, g.obs, g.act)
    d = d.astype(np.float32)
    TOL = 2e-5
    for k in range(g.K):
        idx = g[f"step{k}/idx"]
        e1, e2 = g[f"step{k}/eps1"], g[f"step{k}/eps2"]
        info = o.update(s[idx], a[idx], r[idx], s2[idx], d[idx], e1, e2)
        assert rel_l2(o.last["y"], g[f"step{k}/y"]) < TOL
        assert rel_l2(o.last["lp"], g[f"step{k}/lp"]) < TOL
        assert rel_l2(o.last["q1"], g[f"step{k}/q1"]) < TOL
        assert abs(float(o.last["q1_loss"]) - float(g[f"step{k}/q1_loss"])) <= TOL * abs(float(g[f"step{k}/q1_loss"]))
        cg = o.last["critic_grads"]
        for tag, key in (("q1", "gq1"), ("q2", "gq2")):
            ref = g.sd(f"step{k}/{key}")
            mine = _flat_grads(cg[tag]["dW"], cg[tag]["db"])
            for nm in ref:
                assert rel_l2(mine[nm], ref[nm]) < 5e-5, (k, tag, nm)
        ag = o.last["actor_grads"]
        ref = g.sd(f"step{k}/gpi")
        mine = _flat_grads(ag["dW"], ag["db"])
        for nm in ref:
            assert rel_l2(mine[nm], ref[nm]) < 5e-5, (k, "pi", nm)
        if g.cfg["sac"]["auto_entropy_tuning"]:
            assert abs(float(o.log_alpha) - float(g[f"step{k}/log_alpha"])) < 1e-6
            assert abs(info["alpha_loss"] - float(g[f"step{k}/alpha_loss"])) < 1e-5 * max(1, abs(float(g[f"step{k}/alpha_loss"])))
        for tag in ("pi", "q1", "q2", "q1t", "q2t"):
            ref = g.sd(f"step{k}/{tag}")
            mine = mlp_to_state_dict(getattr(o, tag))
            for nm in ref:
                # Adam's first steps are lr*sign(g): elements whose gradient is at noise level may flip,
                # so compare parameters with a norm-relative metric (SURVEY 7.3 item 3)
                assert rel_l2(mine[nm], ref[nm]) < 1e-4, (k, tag, nm)
        # teacher forcing: continue from the reference's exact post-update state
        for tag, cfgk in (("pi", "policy_net"), ("q1", "q_net"), ("q2", "q_net"), ("q1t", "q_net"), ("q2t", "q_net")):
            net = mlp_from_state_dict(g.sd(f"step{k}/{tag}"), g.cfg[cfgk]["hidden_layers_act"], g.cfg[cfgk]["output_activation"])
            cur = getattr(o, tag)
            for w_dst, w_src in zip(cur.tensors(), net.tensors()):
                w_dst[...] = w_src


@pytest.mark.parametrize("name", ["tiny_auto", "acts_gelu"])
def test_numpy_oracle_adam_state(name):
    """Free-running K updates; Adam moments after K steps match the reference's optimiser state."""
    g = Golden(name)
    o = numpy_oracle_from_golden(g)
    s, a, r, s2, d = synth_transitions(g.n_fill, g.obs, g.act)
    d = d.astype(np.float32)
    for k in range(g.K):
        idx = g[f"step{k}/idx"]
        o.update(s[idx], a[idx], r[idx], s2[idx], d[idx], g[f"step{k}/eps1"], g[f"step{k}/eps2"])
    ad = g.sd(f"step{g.K - 1}/adam_pi")
    for i, (m, v) in enumerate(zip(o.opt_pi.m, o.opt_pi.v)):
        assert rel_l2(m, ad[f"{i}.exp_avg"]) < 1e-4
        assert rel_l2(v, ad[f"{i}.exp_avg_sq"]) < 1e-4
        assert float(ad[f"{i}.step"]) == g.K


def test_numpy_oracle_fp64_twin_noise_floor():
    """fp64 twin of the same math: the fp32 oracle and the fp32 reference sit equally far from it."""
    g = Golden("tiny_auto")
    o32 = numpy_oracle_from_golden(g, np.float32)
    o64 = numpy_oracle_from_golden(g, np.float64)
    s, a, r, s2, d = synth_transitions(g.n_fill, g.obs, g.act)
    idx = g["step0/idx"]
    for o, dt in ((o32, np.float32), (o64, np.float64)):
        o.update(s[idx].astype(dt), a[idx].astype(dt), r[idx].astype(dt), s2[idx].astype(dt),
                 d[idx].astype(dt), g["step0/eps1"].astype(dt), g["step0/eps2"].astype(dt))
    ref_y = g["step0/y"]
    e_ref = rel_l2(ref_y, o64.last["y"])
    e_np = rel_l2(o32.last["y"], o64.last["y"])
    assert e_ref < 1e-5 and e_np < 1e-5


def test_select_action_golden():
    for name in ("tiny_auto", "acts_selu", "outact_tanh"):
        g = Golden(name)
        o = numpy_oracle_from_golden(g)
        # load the final recorded policy
        from oracle.sac_numpy import mlp_from_state_dict
        o.pi = mlp_from_state_dict(g.sd(f"step{g.K - 1}/pi"), g.cfg["policy_net"]["hidden_layers_act"],
                                   g.cfg["policy_net"]["output_activation"])
        st = g["act/state"][None, :]
        assert rel_l2(o.act(st, deterministic=True)[0], g["act/deterministic"]) < 1e-5
        assert rel_l2(o.act(st, eps=g["act/eps"])[0], g["act/stochastic"]) < 1e-5


@pytest.mark.parametrize("name", ["cfg3_pendulum256", "ckpt_tiny_auto", "ckpt_pendulum128"])
def test_reference_run_helper_is_bit_exact(name):
    """tests/helpers.py::ReferenceRun (the full-tensor stand-in for the reference used by the GPU suite) in strict mode."""
    from helpers import ReferenceRun
    g = Golden(name)
    ref = ReferenceRun(g, strict=True)
    for _ in range(g.K):
        r = ref.step()
        assert r["mid"] is not None and set(r["after"]) >= {"pi", "q1", "q2", "q1t", "q2t", "adam", "alpha"}
