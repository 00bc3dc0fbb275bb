"""-m gpu: every agent of a population update (n_agents > 1) against the float64 NumPy oracle, on the FFMA population kernel
(sacx_run_kernel with its agent loop) and on the tensor-core population path (3-D tensor maps, per-agent dW scratch and reduce,
the light row kernel at grid (gx, n_agents), the persistent kernel with tc_skip).

Same method and bars as test_gpu_tiles_oracle.py (tests/update_oracle.py), applied to each agent after one launch for all of
them: every agent's per-update scratch NaN before each launch, the gather and Polyak in bits, gradients recovered from m = 0
with `g.*` left untouched, the critics' batch off every discontinuity of that agent's own nets, two K = 1 launches per case.

Agents differ in everything the kernels index by agent, so an agent that reads another's data fails its own oracle: nets and
targets, Adam v, step counts (0 / 1 / 39 886 mixed per optimiser), log_alpha and its moments, gamma, tau, the temperature's
and three different optimisers' learning rates in the scalar block (some left at 0: the config's value), the update counter,
the device RNG seed, the ring fill (wrapped, partly filled, exactly full, with different push counts) and the batch.

Beyond the per-agent oracle: a perturbed agent leaves every other agent's bits alone; a K = 3 launch equals three K = 1
launches (the (step, agent) indexing of the external batch arrays); act / act_population / q_values against the float64
policy and critics with the agents' own device noise streams.
"""
import numpy as np
import pytest
import torch

from gpu_helpers import base_config, dev, load_nets
from helpers import rel_l2
from test_gpu_parity import _random_nets
from update_oracle import F32, SWITCHES, T, _np, _poison, case, check_update, prepare, report

pytestmark = pytest.mark.gpu

ROWS_PER_TILE = 8                            # rows of one row-op tile (one per warp of a 256-thread CTA)
MAX_CTAS_PER_SM = 8                          # 2048 threads per SM / 256: the light row kernel's occupancy cannot exceed it
FILLS = ("wrapped", "partial", "full")       # agent ag's ring: FILLS[ag % 3]; CTAs that run two agents see different fills
D128 = ((128, 128), (128, 128))


def pop(c, n, tc, what, ctas=0, base=0):
    """n: agents, or a function of the SM count."""
    return dict(c=c, n=n, tc=tc, what=what, ctas=ctas, base=base)


# id: population case, tensor-core path expected, what it reaches
CASES = {
    "ffma-basic": pop(case(24, 4, (256, 256), (256, 256), 96), 5, False, "one agent per CTA, 64x64 tiles"),
    "ffma-loop-default": pop(case(5, 2, (32, 32), (32, 32), 24), lambda sms: sms + 3, False,
                             "grid_y = n_sms: CTAs 0-2 run a second agent (agent loop, gather cache keyed by agent)"),
    "ffma-loop-coop": pop(case(11, 3, (64, 64), (64, 64), 64), 5, False,
                          "64 CTAs per agent, grid_y = 2: cooperative, one barrier counter per group carried across agents, "
                          "last_agent skips the final barrier", ctas=64),
    "ffma-ragged": pop(case(7, 5, (33, 17), (19, 23), 50, actfn="tanh", scale=2.5, lo=-1.0, hi=0.3), 6, False,
                       "odd widths, nothing 16-byte aligned, action_scale 2.5, active log-std clamp"),
    "ffma-saved-z": pop(case(24, 4, (64, 64), (64, 64), 80, actfn="elu", out_act="tanh"), 4, False,
                        "elu hidden, tanh output: saved pre-activations"),
    "ffma-fixed-alpha": pop(case(12, 3, (64, 48), (48, 64), 72, auto=False), 5, False, "fixed temperature, per-agent alpha"),
    "tc-default": pop(case(24, 4, *D128, 256), 64, True, "default threshold: 64 x 256 = 4 x 4096 rows"),
    "tc-b200": pop(case(24, 4, *D128, 200, lo=-1.0, hi=0.3, env={"SACX_TC_MIN_BATCH": "128"}), 3, True,
                   "second 128-row tile of every agent holds 72 rows; active clamp"),
    "tc-b129": pop(case(24, 4, *D128, 129, env={"SACX_TC_MIN_BATCH": "128"}), 4, True,
                   "second 128-row tile of every agent holds one row"),
    "tc-warp-rows-many": pop(case(8, 2, (64, 64), (64, 64), 512, env={"SACX_TC_HEADS": "0", "SACX_TC_ROWS": "0"}), 256, True,
                             "light row kernel: a CTA walks several tiles of one agent, staged head weights reused"),
    "tc-mixed": pop(case(20, 3, (512, 12, 250), (64, 254), 256, env={"SACX_TC_MIN_BATCH": "256"}), 4, True,
                    "512-wide layer and dA N = 12 on FFMA: persistent kernel with tc_skip at grid (grid_x, grid_y)"),
    "devrng-ffma": pop(case(17, 3, (48, 40), (40, 48), 70, actfn="tanh", device_rng=True), 5, False,
                       "device indices and normals, rng_agent = 3 + agent, per-agent seeds", base=3),
    "devrng-tc": pop(case(24, 4, *D128, 256, actfn="tanh", device_rng=True, env={"SACX_TC_MIN_BATCH": "256"}), 4, True,
                     "device indices and OP_PI_TAIL normals, rng_agent = 3 + agent, per-agent seeds", base=3),
}


def _n_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ------------------------------------------------------------------------------------------------------------- set-up
def setup_population(p, monkeypatch, seed, perturb=None):
    """Engine and ring of a population whose agents differ in every agent-indexed input; agent `perturb` draws all of its
    own (weights, ring rows, batch, scalars) from another stream. Returns (eng, rb, rings, rngs): rings[ag] the agent's
    logical ring positions as (s, a, r, s2, d), rngs[ag] the stream its batches are drawn from."""
    from sac.engine import UpdateEngine
    from sac.replay_buffer import ReplayBuffer
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    c = p["c"]
    for k, v in c["env"].items():
        monkeypatch.setenv(k, v)
    n = p["n"](_n_sms()) if callable(p["n"]) else p["n"]
    O, A, B = c["obs"], c["act"], c["B"]
    cap = max(3 * B, 200)
    cfg = base_config(hidden=c["hp"], q_hidden=c["hq"], act=c["actfn"], out_act=c["out_act"], auto=c["auto"], batch=B,
                      seed=seed, capacity=cap, alpha=0.13, log_std_min=c["lo"], log_std_max=c["hi"], action_scale=c["scale"])
    eng = UpdateEngine(O, A, cfg, n_agents=n, ctas_per_agent=p["ctas"], agent_id_base=p["base"])
    eng.reset_state()                     # before the per-agent state: it copies the critics into the targets
    rb = ReplayBuffer(cap, O, A, n_agents=n)
    rings, rngs = [], []
    nl = len(c["hp"])
    for ag in range(n):
        rng = np.random.default_rng([seed, ag] + ([1] if ag == perturb else []))
        sds = _random_nets(O, A, c["hp"], c["hq"], seed=int(rng.integers(2 ** 31)), scale=0.15)
        for nm in (f"net.{2 * nl}.weight", f"net.{2 * nl}.bias"):      # moderate policy heads (update_oracle.setup)
            sds["pi"][nm] = sds["pi"][nm] * F32(0.25)
        for tag in ("q1", "q2"):
            sds[tag + "t"] = {k: (v * (1 + 0.05 * rng.standard_normal(v.shape))).astype(F32) for k, v in sds[tag].items()}
        load_nets(eng, sds, agent=ag)
        eng.view("block.m", ag).zero_()
        eng.view("block.v", ag).copy_(torch.as_tensor(rng.uniform(1e-8, 1e-6, eng.view("block.v", ag).shape).astype(F32)))
        eng.view("scal.step", ag).copy_(torch.tensor([T[(ag + o) % 3] for o in range(4)], dtype=torch.int64))
        eng.view("scal.log_alpha", ag).fill_(float(np.log(0.13) + 0.3 * rng.standard_normal()))
        eng.view("scal.alpha_m", ag).fill_(float(0.01 * rng.standard_normal()))
        eng.view("scal.alpha_v", ag).fill_(float(rng.uniform(1e-3, 1e-1)))
        if not c["auto"]:
            eng.view("scal.alpha", ag).fill_(float(F32(rng.uniform(0.05, 0.3))))
        # trial hyper-parameters as SACPopulation.set_trial writes them; every fifth agent keeps the config's learning rate
        # for Q2 and for the temperature (0 in the scalar block)
        lr = rng.uniform(1e-4, 1e-3, 3)
        if ag % 5 == 4:
            lr[2] = 0.0
        eng.view("scal.lr", ag).copy_(torch.as_tensor(lr))
        eng.view("scal.alpha_lr", ag).fill_(0.0 if ag % 5 == 4 else float(rng.uniform(1e-4, 1e-3)))
        tau = float(rng.uniform(0.001, 0.05))
        eng.view("scal.tau", ag).copy_(torch.as_tensor([F32(tau), F32(1.0 - tau)]))
        eng.view("scal.gamma", ag).fill_(float(F32(rng.uniform(0.9, 0.999))))
        eng.view("scal.updates", ag).fill_(int(rng.integers(0, 100000)))
        eng.view("scal.rng_seed", ag).fill_(int(rng.integers(1, 2 ** 62)))
        kind = FILLS[ag % 3]
        n_push = {"wrapped": cap + cap // 3 + 7 + 13 * (ag % 5), "partial": cap - 5 - 3 * (ag % 5), "full": cap}[kind]
        s = rng.standard_normal((n_push, O)).astype(F32)
        s2 = rng.standard_normal((n_push, O)).astype(F32)
        a = rng.uniform(-1, 1, (n_push, A)).astype(F32)
        r = rng.standard_normal(n_push).astype(F32)
        d = (rng.random(n_push) < 0.4).astype(F32)
        for lo in range(0, n_push, cap // 2):
            sl = slice(lo, lo + cap // 2)
            rb.push_batch(s[sl], a[sl], r[sl], s2[sl], d[sl], agent=ag)
        first = max(n_push - cap, 0)
        rings.append(tuple(x[first:] for x in (s, a, r, s2, d)))
        rngs.append(rng)
    eng.refresh_alpha()
    eng.attach_ring(rb)
    return eng, rb, rings, rngs


def _launch(eng, c, us):
    """One K = 1 update of every agent from its prepared batch (device RNG: the kernels draw it)."""
    n = eng.n_agents
    for ag in range(n):
        _poison(eng, ag)
    if c["device_rng"]:
        eng.update(None, None, None, 1)
    else:
        eng.update(*(dev(np.stack([u[k] for u in us])[None]) for k in ("idx", "e1", "e2")), 1)
    eng.sync()


def _check_path(eng, p, tc_before=None):
    kind, why = eng.path()
    assert kind == "tiles", (kind, why)
    on, tc_why, launches = eng.tensor_core()
    assert on == p["tc"], tc_why
    if tc_before is not None:
        assert (launches > tc_before) == p["tc"], (launches, tc_before)
    return launches


def _check_grid(name, eng, p):
    gx, gy, _ = eng.grid()
    n, sms = eng.n_agents, _n_sms()
    assert (gx, gy) == (max(1, p["ctas"]), min(n, sms // max(1, p["ctas"]))), (gx, gy)
    if name.startswith("ffma-loop"):
        assert n > gy, "the case must reach the agent loop"
    if name == "ffma-loop-default":
        assert gy == sms
    if name == "ffma-loop-coop":
        assert (gx, gy) == (64, 2)
    if name == "tc-warp-rows-many":
        # light row kernel: gx = min(tiles, ceil(8 slots / n)), slots = n_sms x CTAs per SM
        gx_max = -(-8 * sms * MAX_CTAS_PER_SM // n)
        assert -(-p["c"]["B"] // ROWS_PER_TILE) > gx_max, "a CTA must walk several tiles of one agent"
    return gx, gy


# ------------------------------------------------------------------------------------------------------------- per agent
@pytest.mark.parametrize("name", list(CASES))
def test_population_update_vs_float64_oracle(name, monkeypatch):
    p = CASES[name]
    c = p["c"]
    eng, rb, rings, rngs = setup_population(p, monkeypatch, 4000 + 17 * c["obs"] + c["act"])
    grid = _check_grid(name, eng, p)
    launches = _check_path(eng, p)
    worst, flagged = {}, []
    for k in range(2):
        if k:
            for ag in range(eng.n_agents):
                eng.view("block.m", ag).zero_()
        us = [prepare(eng, c, rings[ag], rngs[ag], agent=ag) for ag in range(eng.n_agents)]
        _launch(eng, c, us)
        launches = _check_path(eng, p, launches)
        fl = [check_update(eng, c, rings[ag], us[ag], eng.metrics(ag), worst, agent=ag) for ag in range(eng.n_agents)]
        flagged.append(tuple(int(sum(f[i] for f in fl)) for i in range(2)))
    report(f"{name}: {'tensor core' if p['tc'] else 'FFMA'} population, {eng.n_agents} agents, grid {grid}: {p['what']}",
           c, flagged, worst)


# ------------------------------------------------------------------------------------------------------------- isolation
def _snapshot(eng, ag):
    """Bits of an agent's parameters, targets, Adam moments, gradients, outputs and scalar block."""
    return {k: _np(eng.view(k, ag)).view(np.uint8) for k in eng.layout if k.startswith(("block.", "out.", "scal."))}


def _draw(eng, p, rings, rngs, K):
    c = p["c"]
    B, A = c["B"], c["act"]
    idx = np.stack([np.stack([rngs[ag].choice(len(rings[ag][0]), B, replace=False) for ag in range(eng.n_agents)])
                    for _ in range(K)]).astype(np.int64)
    e1, e2 = (np.stack([rngs[ag].standard_normal((K, B, A)) for ag in range(eng.n_agents)], axis=1).astype(F32) for _ in range(2))
    return idx, e1, e2


@pytest.mark.parametrize("name", ["ffma-loop-default", "tc-b200"])
def test_population_agent_perturbation_leaves_other_agents_bits(name, monkeypatch):
    """The case built twice from the same seeds, the second time with agent 1's weights, ring rows, batch and scalars drawn
    from another stream: one update of each, every other agent bit-identical. On ffma-loop-default agent 1 shares CTA 1 with
    agent n_sms + 1, which runs after it."""
    p, k = CASES[name], 1
    snaps = []
    for perturb in (None, k):
        eng, rb, rings, rngs = setup_population(p, monkeypatch, 77, perturb)
        idx, e1, e2 = _draw(eng, p, rings, rngs, 1)
        for ag in range(eng.n_agents):
            _poison(eng, ag)
        eng.update(dev(idx), dev(e1), dev(e2), 1)
        eng.sync()
        snaps.append([_snapshot(eng, ag) for ag in range(eng.n_agents)])
        del eng, rb
    for ag in range(len(snaps[0])):
        same = [nm for nm in snaps[0][ag] if np.array_equal(snaps[0][ag][nm], snaps[1][ag][nm])]
        if ag == k:
            assert "block.params" not in same, "the perturbation did not reach agent k"
        else:
            assert len(same) == len(snaps[0][ag]), f"agent {ag}: {sorted(set(snaps[0][ag]) - set(same))} changed with agent {k}"


# ------------------------------------------------------------------------------------------------------------- multi-step
@pytest.mark.parametrize("name", ["ffma-loop-coop", "tc-b200"])
def test_population_multi_step_launch_equals_single_steps(name, monkeypatch):
    """update(idx[3, n, B], eps1, eps2, 3) against three K = 1 launches, bit for bit for every agent: step s of agent ag reads
    row (s n + ag) of the external arrays."""
    p, K = CASES[name], 3
    snaps = []
    for single in (True, False):
        eng, rb, rings, rngs = setup_population(p, monkeypatch, 91)
        _check_path(eng, p)
        upd0 = [eng.metrics(ag)["updates"] for ag in range(eng.n_agents)]
        idx, e1, e2 = _draw(eng, p, rings, rngs, K)
        if single:
            for s in range(K):
                eng.update(dev(idx[s:s + 1]), dev(e1[s:s + 1]), dev(e2[s:s + 1]), 1)
        else:
            eng.update(dev(idx), dev(e1), dev(e2), K)
        eng.sync()
        for ag in range(eng.n_agents):
            m = eng.metrics(ag)
            assert m["updates"] == upd0[ag] + K and m["nonfinite"] == 0
        snaps.append([_snapshot(eng, ag) for ag in range(eng.n_agents)])
        del eng, rb
    for ag in range(len(snaps[0])):
        diff = [nm for nm in snaps[0][ag] if not np.array_equal(snaps[0][ag][nm], snaps[1][ag][nm])]
        assert not diff, f"agent {ag}: K = {K} launch differs from {K} single launches in {diff}"


# ------------------------------------------------------------------------------------------------------------- acting
def test_population_act_and_q_values_vs_float64(monkeypatch):
    """act_population and act(agent = k) on distinct agents (agent_id_base 3): deterministic and given-noise actions and
    q_values(agent = k) against the float64 networks of agent k; device noise from the agent's own stream
    philox_normal(seed_k, act call, 3, row, j, 3 + k), checked through the actions."""
    from oracle import device_rng
    from oracle.sac_numpy import squash_sample
    from update_oracle import _mlp, _state
    p = pop(case(7, 5, (33, 17), (19, 23), 50, actfn="tanh", scale=2.5, lo=-1.0, hi=0.3), 8, False, "acting", base=3)
    c = p["c"]
    eng, rb, rings, rngs = setup_population(p, monkeypatch, 55)
    n, O, A, rows = eng.n_agents, c["obs"], c["act"], 6
    rng = np.random.default_rng(56)
    nets = [_state(eng, c, ag) for ag in range(n)]
    pis = [_mlp(st["pi"], c["actfn"], c["out_act"]) for st in nets]
    states = rng.standard_normal((n, rows, O)).astype(F32)
    heads = [pis[ag].forward(states[ag].astype(np.float64))[0] for ag in range(n)]
    seeds = [int(eng.view("scal.rng_seed", ag).item()) for ag in range(n)]
    assert len(set(seeds)) == n
    counter = int(eng.lib.sacx_agent_act_counter(eng.h, -1))
    worst = {}

    def bar(what, e, lim=2e-5):
        worst[what] = max(worst.get(what, 0.0), e)
        assert e < lim, f"{what}: {e:.3e} >= {lim:.1e}"

    def normals(ag, cnt):
        return np.array([[device_rng.philox_normal(seeds[ag], cnt, 3, row, j, p["base"] + ag) for j in range(A)]
                         for row in range(rows)])

    def device_noise(ag, got, e_ref, given):
        """got: actions drawn with the device noise; given: the same kernel on the float32 normals e_ref of that call. The
        device's normals may differ from e_ref by a few ulps, which moves an action by at most |da/de| x those ulps plus the
        rounding of z and of the action."""
        ref, _, aux = squash_sample(heads[ag], e_ref, c["lo"], c["hi"], c["scale"])
        bar("act device noise", rel_l2(got, ref))
        sd = np.exp(np.clip(heads[ag][:, A:], c["lo"], c["hi"]))
        dtz = c["scale"] * (1 - aux["tz"] ** 2)
        slack = dtz * 2 * np.spacing(np.abs(aux["z"]).astype(F32)) + 2 * np.spacing(np.abs(ref).astype(F32))
        ulps = np.maximum(np.abs(got - given) - slack, 0) / (dtz * sd * np.spacing(F32(1)) * np.maximum(1.0, np.abs(e_ref)))
        bar("act device normals (ulps)", float(ulps.max()), 4.0 + 1e-9)

    # ---- act_population: one launch, grid (rows, agents)
    a = _np(eng.act_population(dev(states), deterministic=True)); counter += 1
    for ag in range(n):
        bar("act deterministic", rel_l2(a[ag], np.tanh(heads[ag][:, :A]) * c["scale"]))
    eps = rng.standard_normal((n, rows, A)).astype(F32)
    a = _np(eng.act_population(dev(states), eps=dev(eps))); counter += 1
    for ag in range(n):
        bar("act given eps", rel_l2(a[ag], squash_sample(heads[ag], eps[ag].astype(np.float64), c["lo"], c["hi"], c["scale"])[0]))
    a = _np(eng.act_population(dev(states)))
    e_ref = np.stack([normals(ag, counter) for ag in range(n)])
    counter += 1
    given = _np(eng.act_population(dev(states), eps=dev(e_ref.astype(F32)))); counter += 1
    for ag in range(n):
        device_noise(ag, a[ag], e_ref[ag], given[ag])

    # ---- act(agent = k): one agent, grid (rows, 1)
    for ag in range(n):
        s = dev(states[ag])
        bar("act deterministic", rel_l2(_np(eng.act(s, deterministic=True, agent=ag)), np.tanh(heads[ag][:, :A]) * c["scale"]))
        bar("act given eps", rel_l2(_np(eng.act(s, eps=dev(eps[ag]), agent=ag)),
                                    squash_sample(heads[ag], eps[ag].astype(np.float64), c["lo"], c["hi"], c["scale"])[0]))
        got = _np(eng.act(s, agent=ag))
        e_ref = normals(ag, counter + 2)
        given = _np(eng.act(s, eps=dev(e_ref.astype(F32)), agent=ag))
        counter += 4
        device_noise(ag, got, e_ref, given)
    assert int(eng.lib.sacx_agent_act_counter(eng.h, -1)) == counter

    # ---- q_values(agent = k)
    acts = rng.uniform(-1, 1, (rows, A)).astype(F32)
    for ag in range(n):
        q1, q2 = eng.q_values(dev(states[ag]), dev(acts), agent=ag)
        x = np.concatenate([states[ag], acts], axis=1).astype(np.float64)
        for got, tag in ((q1, "q1"), (q2, "q2")):
            bar("q_values", rel_l2(_np(got), _mlp(nets[ag][tag], c["actfn"], c["out_act"]).forward(x)[0][:, 0]))
    print(f"\n[act / q_values] {n} agents x {rows} rows, agent_id_base {p['base']}, {counter} act calls")
    for q, e in sorted(worst.items()):
        print(f"    {q:34s} {e:.2e}")
