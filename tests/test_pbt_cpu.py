"""Population-based training's host logic without a device (sac/pbt.py): truncation selection, explore, the hyper-parameter
records against SACPopulation.set_trial's roundings, the cross-rank routing of an exploit, and refused pair lists."""
import ctypes
import types

import numpy as np
import pytest
import torch

from sac import _engine as E
from sac.pbt import PBTConfig, check_pairs, explore, pbt_record, round_rng, route_exploit, select_pairs
from sac.population import SACPopulation, shard_agents

SPACE = {"sac": {"alpha": {"type": "loguniform", "low": 0.01, "high": 0.5},
                 "alpha_lr": {"type": "loguniform", "low": 1e-4, "high": 1e-2},
                 "tau": {"type": "uniform", "low": 0.001, "high": 0.05},
                 "gamma": {"type": "categorical", "choices": [0.95, 0.99]}}}


# ------------------------------------------------------------------------------------------------------------- selection
def test_selection_bottom_receives_from_top():
    scores = [float(s) for s in [5, 1, 9, 3, 7, 2, 8, 0, 6, 4]]
    pairs = select_pairs(scores, 0.2, round_rng(0, 0))
    assert [d for _, d in pairs] == [1, 7]                       # the two lowest, in id order
    assert all(s in (2, 6) for s, _ in pairs)                    # from the two highest
    assert select_pairs(scores, 0.2, round_rng(0, 0)) == pairs   # deterministic for (seed, round)
    draws = {tuple(select_pairs(scores, 0.3, round_rng(3, r))) for r in range(20)}
    assert len(draws) > 1                                        # the source is drawn, not fixed
    for ps in draws:
        assert [d for _, d in ps] == [1, 5, 7] and all(s in (2, 6, 4) for s, _ in ps)


def test_selection_top_set_is_uniform_and_fixed_size():
    scores = [float(g) for g in range(10)]
    seen = set()
    for r in range(200):
        ps = select_pairs(scores, 0.3, round_rng(1, r))
        assert [d for _, d in ps] == [0, 1, 2]
        seen |= {s for s, _ in ps}
    assert seen == {7, 8, 9}


def test_selection_ties_break_by_global_id():
    scores = [1.0] * 6
    ps = select_pairs(scores, 0.34, round_rng(0, 0))             # k = 2: the lower id ranks higher
    assert [d for _, d in ps] == [4, 5] and all(s in (0, 1) for s, _ in ps)


def test_selection_eligibility_and_finished_trials():
    scores = [None, 3.0, None, 1.0, 2.0, None, 0.5, 4.0, None, None]   # None: finished or too few episodes
    ps = select_pairs(scores, 0.5, round_rng(0, 1))
    assert [d for _, d in ps] == [3, 6] and all(s in (1, 7) for s, _ in ps)
    assert select_pairs([None] * 4 + [1.0], 0.5, round_rng(0, 0)) == []
    assert select_pairs([1.0, 2.0, 3.0, 4.0], 0.2, round_rng(0, 0)) == []       # floor(0.8) = 0


def test_config_refusals():
    with pytest.raises(ValueError):
        PBTConfig(0)
    with pytest.raises(ValueError):
        PBTConfig(10, fraction=0.6)
    with pytest.raises(ValueError):
        PBTConfig(10, perturb=(0.0, 1.2))
    with pytest.raises(ValueError):
        PBTConfig(10, resample_probability=1.5)
    with pytest.raises(ValueError):
        PBTConfig(10, min_episodes=0)


# ------------------------------------------------------------------------------------------------------------- explore
def test_explore_perturbs_by_the_factors_and_clips():
    cfg = PBTConfig(10, perturb=(0.8, 1.2), resample_probability=0.0)
    vals = {"sac.alpha_lr": 1e-3, "sac.tau": 0.01, "sac.actor_lr": 3e-4}
    factors = set()
    for r in range(50):
        out = explore(vals, SPACE, cfg, round_rng(0, r))
        assert list(out) == list(vals)
        for k in ("sac.alpha_lr", "sac.tau", "sac.actor_lr"):
            f = out[k] / vals[k]
            assert min(abs(f - 0.8), abs(f - 1.2)) < 1e-12
            factors.add(round(f, 6))
    assert factors == {0.8, 1.2}
    hi = explore({"sac.tau": 0.049}, SPACE, cfg, round_rng(0, 0))
    lo = explore({"sac.alpha": 0.011}, SPACE, cfg, round_rng(0, 0))
    for _ in range(20):
        assert 0.001 <= explore({"sac.tau": 0.049}, SPACE, cfg, round_rng(5, _))["sac.tau"] <= 0.05
        assert 0.01 <= explore({"sac.alpha": 0.011}, SPACE, cfg, round_rng(5, _))["sac.alpha"] <= 0.5
    assert hi["sac.tau"] in (0.05, 0.049 * 0.8) and lo["sac.alpha"] in (0.011 * 1.2, 0.01)


def test_explore_resamples_within_the_space():
    cfg = PBTConfig(10, resample_probability=1.0)
    outs = [explore({"sac.alpha": 0.1, "sac.tau": 0.01}, SPACE, cfg, round_rng(2, r)) for r in range(30)]
    for o in outs:
        assert 0.01 <= o["sac.alpha"] <= 0.5 and 0.001 <= o["sac.tau"] <= 0.05
    assert len({o["sac.alpha"] for o in outs}) == 30


def test_explore_categorical_keys_redraw_or_stay():
    stay = PBTConfig(10, resample_probability=0.0)
    assert all(explore({"sac.gamma": 0.95}, SPACE, stay, round_rng(0, r))["sac.gamma"] == 0.95 for r in range(20))
    redraw = PBTConfig(10, resample_probability=1.0)
    got = {explore({"sac.gamma": 0.95}, SPACE, redraw, round_rng(0, r))["sac.gamma"] for r in range(40)}
    assert got == {0.95, 0.99}


def test_explore_refuses_keys_outside_the_trial_keys():
    cfg = PBTConfig(10)
    for key in ("train.batch_size", "q_net.hidden_sizes", "sac.auto_entropy_tuning"):
        with pytest.raises(ValueError, match="cannot be explored"):
            explore({key: 1}, SPACE, cfg, round_rng(0, 0))


def test_explore_is_deterministic():
    cfg = PBTConfig(10)
    v = {"sac.alpha": 0.1, "sac.alpha_lr": 1e-3, "sac.gamma": 0.99}
    assert explore(v, SPACE, cfg, round_rng(4, 7)) == explore(v, SPACE, cfg, round_rng(4, 7))


# ------------------------------------------------------------------------------------------------------------- records
class _FakeEngine:
    """The scalar-block views SACPopulation.set_trial writes, as host tensors of the engine's dtypes."""

    def __init__(self):
        self.t = {"scal.log_alpha": torch.zeros(1, dtype=torch.float64), "scal.alpha": torch.zeros(1, dtype=torch.float64),
                  "scal.alpha_lr": torch.zeros(1, dtype=torch.float64), "scal.lr": torch.zeros(3, dtype=torch.float64),
                  "scal.tau": torch.zeros(1, 2, dtype=torch.float32), "scal.gamma": torch.zeros(1, 1, dtype=torch.float32),
                  "scal.alpha_f32": torch.zeros(1, 1, dtype=torch.float32)}

    def view(self, name, agent=0):
        return self.t[name]

    def sync(self):
        pass

    def refresh_alpha(self):              # sacx_agent_refresh_alpha with a fixed temperature
        self.t["scal.alpha_f32"].fill_(float(self.t["scal.alpha"].item()))


@pytest.mark.parametrize("vals", [
    {"alpha": 0.1234567, "alpha_lr": 3.3e-4, "actor_lr": 1.0e-3 / 3, "critic_lr": 7.7e-4, "tau": 0.0051, "gamma": 0.987654321},
    {"alpha": 0.7, "tau": 0.3},
    {"tau": 1.0, "gamma": 1.0},
    {"critic_lr": 0.1},
])
def test_records_equal_set_trials_roundings(vals):
    fake = _FakeEngine()
    SACPopulation.set_trial(types.SimpleNamespace(engine=fake, config={"sac": {"auto_entropy_tuning": False}}), 0, **vals)
    r = pbt_record(vals, auto_alpha=False)
    f32 = lambda x: np.float32(x).tobytes()         # noqa: E731
    f64 = lambda x: np.float64(x).tobytes()         # noqa: E731
    if "alpha" in vals:
        assert r.set & E.PBT_ALPHA
        assert f64(r.log_alpha) == f64(fake.t["scal.log_alpha"].item()) and f64(r.alpha) == f64(fake.t["scal.alpha"].item())
        assert f32(r.alpha_f32) == f32(fake.t["scal.alpha_f32"].item())
    if "alpha_lr" in vals:
        assert f64(r.alpha_lr) == f64(fake.t["scal.alpha_lr"].item())
    lr = fake.t["scal.lr"].tolist()
    if "actor_lr" in vals:
        assert f64(r.actor_lr) == f64(lr[0])
    if "critic_lr" in vals:
        assert f64(r.critic_lr) == f64(lr[1]) == f64(lr[2])
    if "tau" in vals:
        t = fake.t["scal.tau"].reshape(-1).tolist()
        assert f32(r.tau) == f32(t[0]) and f32(r.one_minus_tau) == f32(t[1])
    if "gamma" in vals:
        assert f32(r.gamma) == f32(fake.t["scal.gamma"].item())
    want = sum(bit for k, bit in (("alpha", E.PBT_ALPHA), ("alpha_lr", E.PBT_ALPHA_LR), ("actor_lr", E.PBT_ACTOR_LR),
                                  ("critic_lr", E.PBT_CRITIC_LR), ("tau", E.PBT_TAU), ("gamma", E.PBT_GAMMA)) if k in vals)
    assert r.set == want


def test_record_one_minus_tau_is_rounded_once_from_double():
    tau = 0.1 + 1e-9
    assert pbt_record({"tau": tau}, False).one_minus_tau == float(np.float32(1.0 - tau))


def test_record_with_auto_temperature_never_writes_alpha():
    r = pbt_record({"alpha": 0.2, "alpha_lr": 1e-3}, auto_alpha=True)
    assert r.set == E.PBT_ALPHA_LR and r.alpha == 0.0 and r.log_alpha == 0.0
    assert pbt_record(None, True).set == 0 and pbt_record({}, False).set == 0


def test_record_refusals():
    for bad in ({"alpha": 0.0}, {"actor_lr": -1e-3}, {"critic_lr": float("nan")}, {"gamma": float("inf")}, {"tau": 0.0},
                {"tau": 1.5}, {"alpha_lr": -0.0}):
        with pytest.raises(ValueError):
            pbt_record(bad, False)
    with pytest.raises(KeyError):
        pbt_record({"batch_size": 3}, False)


def test_record_mirrors_the_library_struct():
    assert E.SacxPbtRecord.set.offset == 0
    assert E.SacxPbtRecord.log_alpha.offset == 8 and E.SacxPbtRecord.alpha_f32.offset == 48
    assert ctypes.sizeof(E.SacxPbtRecord) == 64


# ------------------------------------------------------------------------------------------------------------- routing
def _emulate(pairs, n_agents, world, state=None):
    """Carry out the routes on host 'arenas' (one value per agent) and return the agents afterwards."""
    state = list(range(100, 100 + n_agents)) if state is None else list(state)
    routes = route_exploit(pairs, n_agents, world)
    shards = [list(shard_agents(n_agents, world, r)) for r in range(world)]
    arena = [[state[g] for g in shards[r]] for r in range(world)]
    before = [list(a) for a in arena]
    send = [[before[r][a] for a in routes[r].pack] for r in range(world)]
    for r, rt in enumerate(routes):
        assert sum(rt.send_counts) == len(rt.pack)
        for q in range(world):
            assert rt.send_counts[q] == routes[q].recv_counts[r]                 # split sizes agree pairwise
    recv = []
    for r in range(world):                                                       # all_to_all_single: grouped by source rank
        buf = []
        for q in range(world):
            off = sum(routes[q].send_counts[:r])
            buf += send[q][off: off + routes[q].send_counts[r]]
        assert len(buf) == sum(routes[r].recv_counts)
        recv.append(buf)
    for r, rt in enumerate(routes):
        for s, d in zip(rt.copy_src, rt.copy_dst):
            arena[r][d] = before[r][s]
        for slot, d in zip(rt.unpack_slot, rt.unpack_dst):
            arena[r][d] = recv[r][slot]
    return [v for a in arena for v in a], routes


@pytest.mark.parametrize("world", [1, 2, 8])
def test_routing_delivers_every_source_once(world):
    n = 37
    rng = np.random.default_rng(world)
    for trial in range(20):
        ids = rng.permutation(n)
        k = int(rng.integers(1, n // 3))
        dsts, srcs = ids[:k], ids[k:]
        pairs = [(int(rng.choice(srcs[: max(1, k // 2)])), int(d)) for d in dsts]          # sources feed several destinations
        got, routes = _emulate(pairs, n, world)
        want = list(range(100, 100 + n))
        for s, d in pairs:
            want[d] = 100 + s
        assert got == want
        ppair = sorted(i for rt in routes for i in rt.copy_pair + rt.unpack_pair)
        assert ppair == list(range(len(pairs)))                                    # every pair handled exactly once
        own = {g: r for r in range(world) for g in shard_agents(n, world, r)}
        for r, rt in enumerate(routes):                                            # one state per (source, destination rank)
            need = {(s, own[d]) for s, d in pairs if own[s] == r and own[d] != r}
            assert len(rt.pack) == len(need)
            assert rt.send_counts == [sum(1 for _, q in need if q == x) for x in range(world)]
        if world == 1:
            assert all(not rt.pack for rt in routes)


def test_routing_splits_for_a_known_case():
    # 8 agents on 2 ranks: rank 0 owns 0-3, rank 1 owns 4-7
    pairs = [(0, 5), (0, 6), (1, 2), (4, 3), (4, 7)]
    r0, r1 = route_exploit(pairs, 8, 2)
    assert (r0.copy_src, r0.copy_dst, r0.copy_pair) == ([1], [2], [2])
    assert (r1.copy_src, r1.copy_dst, r1.copy_pair) == ([0], [3], [4])                     # agents 4 -> 7 as local 0 -> 3
    assert r0.pack == [0] and r0.send_counts == [0, 1] and r0.recv_counts == [0, 1]        # agent 0 once for both of 5, 6
    assert r1.pack == [0] and r1.send_counts == [1, 0] and r1.recv_counts == [1, 0]
    assert (r0.unpack_slot, r0.unpack_dst, r0.unpack_pair) == ([0], [3], [3])
    assert (r1.unpack_slot, r1.unpack_dst, r1.unpack_pair) == ([0, 0], [1, 2], [0, 1])


@pytest.mark.parametrize("pairs, match", [
    ([(0, 8)], "out of range"), ([(-1, 2)], "out of range"), ([(0, 1), (2, 1)], "destination twice"),
    ([(0, 1), (1, 2)], "both a source and a destination"), ([(3, 3)], "both a source and a destination"),
])
def test_refused_pair_lists(pairs, match):
    with pytest.raises(ValueError, match=match):
        check_pairs(pairs, 8)
    with pytest.raises(ValueError, match=match):
        route_exploit(pairs, 8, 2)


def test_empty_pair_list_routes_nothing():
    for rt in route_exploit([], 5, 2):
        assert not (rt.copy_dst or rt.pack or rt.unpack_dst) and rt.send_counts == [0, 0]
