"""Population-based training (Jaderberg et al., 2017) over a ``SACPopulation``: host logic only.

At fixed intervals the worst trials take over the learner state of the best ones ("exploit", ``SACPopulation.exploit``: one
device launch per rank, plus one collective when ranks are involved) and perturb or redraw their hyper-parameters ("explore").
Everything here is deterministic for a given (seed, round) and is computed identically on every rank, so the ranks agree on
the pairs without exchanging them:

``select_pairs``     truncation selection: the bottom ``fraction`` of the eligible trials each receive from a top-``fraction``
                     trial drawn uniformly
``explore``          perturb (factor from ``perturb``, clipped to the search space) or resample each hyper-parameter
``pbt_record``       the scalar-block values of a set of hyper-parameters, with exactly ``SACPopulation.set_trial``'s roundings
``route_exploit``    who packs, sends, receives and unpacks what for a list of global (source, destination) pairs
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _engine as E
from .population import SACPopulation, shard_agents

TRIAL_KEYS = SACPopulation.TRIAL_KEYS


@dataclass(frozen=True)
class PBTConfig:
    """interval_steps: environment steps between exploit rounds. fraction: share of the eligible trials that receive (the
    bottom) and that give (the top). perturb: the factors a perturbed value is multiplied by (one drawn uniformly).
    resample_probability: chance that a hyper-parameter is redrawn from the search space instead. min_episodes: episodes a
    trial must have finished since its last exploit to take part. seed: with the round number, seeds every draw."""
    interval_steps: int
    fraction: float = 0.2
    perturb: Tuple[float, ...] = (0.8, 1.2)
    resample_probability: float = 0.25
    min_episodes: int = 1
    seed: int = 0

    def __post_init__(self):
        if int(self.interval_steps) != self.interval_steps or self.interval_steps < 1:
            raise ValueError("PBTConfig.interval_steps must be a positive integer")
        if not 0.0 < self.fraction <= 0.5:
            raise ValueError("PBTConfig.fraction must be in (0, 0.5]: the bottom and top sets must not overlap")
        if not self.perturb or not all(f > 0 and math.isfinite(f) for f in self.perturb):
            raise ValueError("PBTConfig.perturb must hold positive finite factors")
        if not 0.0 <= self.resample_probability <= 1.0:
            raise ValueError("PBTConfig.resample_probability must be in [0, 1]")
        if int(self.min_episodes) != self.min_episodes or self.min_episodes < 1:
            raise ValueError("PBTConfig.min_episodes must be an integer >= 1 (a score is a mean over episodes)")


def round_rng(seed: int, rnd: int) -> np.random.Generator:
    """The generator of one exploit round: the same on every rank."""
    return np.random.default_rng([int(seed), int(rnd)])


def select_pairs(scores: Sequence[Optional[float]], fraction: float, rng: np.random.Generator) -> List[Tuple[int, int]]:
    """Truncation selection over global trial ids. scores[g] is None for a trial that does not take part (finished, or too
    few episodes since its last exploit). Trials rank by score, equal scores by global id (the lower id ranks higher);
    the bottom floor(fraction * n_eligible) each receive from a top-fraction trial drawn uniformly. Returns (source,
    destination) pairs in increasing destination order."""
    eligible = [g for g, s in enumerate(scores) if s is not None]
    k = int(math.floor(fraction * len(eligible)))
    if k == 0:
        return []
    order = sorted(eligible, key=lambda g: (-float(scores[g]), g))          # best first
    top, bottom = order[:k], sorted(order[-k:])
    return [(top[int(rng.integers(k))], dst) for dst in bottom]


def _split_key(key: str) -> Tuple[str, str]:
    section, param = key.split(".", 1)
    if section != "sac" or param not in TRIAL_KEYS:
        raise ValueError(f"{key} cannot be explored: only sac.{{{', '.join(TRIAL_KEYS)}}} may differ between the trials of one "
                         "population")
    return section, param


def _draw(spec: dict, rng: np.random.Generator):
    if spec["type"] == "categorical":
        return spec["choices"][int(rng.integers(len(spec["choices"])))]
    if spec["type"] == "uniform":
        return float(rng.uniform(spec["low"], spec["high"]))
    if spec["type"] == "loguniform":
        return float(math.exp(rng.uniform(math.log(spec["low"]), math.log(spec["high"]))))
    raise ValueError(f"unknown search-space type {spec['type']!r}")


def explore(values: Dict[str, Any], search_space: Optional[Dict[str, Dict[str, dict]]], cfg: PBTConfig,
            rng: np.random.Generator) -> Dict[str, Any]:
    """New values for every key of a trial dict (``section.param`` keys, run_search.py format). Per key, in the dict's order:
    with probability resample_probability a fresh draw from the search space; otherwise a numeric value times a factor drawn
    uniformly from cfg.perturb, clipped to the search space's [low, high], and a categorical value stays. A key the search
    space does not name is perturbed and not clipped."""
    out = {}
    for key, value in values.items():
        section, param = _split_key(key)
        spec = (search_space or {}).get(section, {}).get(param)
        resample = rng.random() < cfg.resample_probability
        if spec is not None and resample:
            out[key] = _draw(spec, rng)
        elif spec is not None and spec["type"] == "categorical":
            out[key] = value
        else:
            v = float(value) * float(cfg.perturb[int(rng.integers(len(cfg.perturb)))])
            if spec is not None:
                v = min(max(v, float(spec["low"])), float(spec["high"]))
            out[key] = v
    return out


def pbt_record(hypers: Optional[Dict[str, float]], auto_alpha: bool) -> E.SacxPbtRecord:
    """Scalar-block values of a subset of ``TRIAL_KEYS`` with ``SACPopulation.set_trial``'s roundings: learning rates as
    python doubles, gamma / tau as float32, one_minus_tau = float32(1.0 - tau) with the difference taken in double; with a
    fixed temperature log_alpha = log(alpha), alpha = float32(alpha), alpha_f32. With auto_entropy_tuning the temperature is
    learner state (it travels with the copy), so an ``alpha`` entry is not written."""
    r = E.SacxPbtRecord()
    for key, value in (hypers or {}).items():
        if key not in TRIAL_KEYS:
            raise KeyError(f"not a per-agent hyper-parameter: {key!r} (per-agent: {TRIAL_KEYS})")
        v = float(value)
        if not (v > 0.0 and math.isfinite(v)):
            raise ValueError(f"{key} must be positive and finite, got {value!r}")
        if key == "alpha":
            if auto_alpha:
                continue
            r.set |= E.PBT_ALPHA
            r.log_alpha = math.log(v)
            r.alpha = float(np.float32(v))
            r.alpha_f32 = r.alpha
        elif key == "alpha_lr":
            r.set |= E.PBT_ALPHA_LR
            r.alpha_lr = v
        elif key == "actor_lr":
            r.set |= E.PBT_ACTOR_LR
            r.actor_lr = v
        elif key == "critic_lr":
            r.set |= E.PBT_CRITIC_LR
            r.critic_lr = v
        elif key == "tau":
            if v > 1.0:
                raise ValueError(f"tau must be in (0, 1], got {value!r}")
            r.set |= E.PBT_TAU
            r.tau = float(np.float32(v))
            r.one_minus_tau = float(np.float32(1.0 - v))
        else:
            r.set |= E.PBT_GAMMA
            r.gamma = float(np.float32(v))
    return r


@dataclass
class RankRoute:
    """What one rank does in an exploit. Local ids throughout; `pair_*` index into the caller's pair list (for records)."""
    copy_src: List[int]          # local pairs: one copy launch
    copy_dst: List[int]
    copy_pair: List[int]
    pack: List[int]              # agents packed into the send buffer, grouped by destination rank in rank order
    send_counts: List[int]       # states sent to each rank
    recv_counts: List[int]       # states received from each rank (the receive buffer is grouped by source rank)
    unpack_slot: List[int]       # receive-buffer slot -> local destination
    unpack_dst: List[int]
    unpack_pair: List[int]


def _owner(n_agents: int, world: int) -> List[int]:
    own = [0] * n_agents
    for r in range(world):
        for g in shard_agents(n_agents, world, r):
            own[g] = r
    return own


def check_pairs(pairs: Sequence[Tuple[int, int]], n_agents: int) -> None:
    """ValueError for an id out of range, a repeated destination, or a destination that is also a source."""
    dsts = set()
    for s, d in pairs:
        for g in (s, d):
            if isinstance(g, bool) or int(g) != g or not 0 <= g < n_agents:
                raise ValueError(f"exploit: agent {g!r} out of range [0, {n_agents})")
        if d in dsts:
            raise ValueError(f"exploit: agent {d} is a destination twice")
        dsts.add(d)
    for s, _ in pairs:
        if s in dsts:
            raise ValueError(f"exploit: agent {s} is both a source and a destination")


def route_exploit(pairs: Sequence[Tuple[int, int]], n_agents: int, world: int) -> List[RankRoute]:
    """The routes of every rank for global (source, destination) pairs, agents sharded by ``shard_agents``. A pair whose
    two agents live on one rank is a local copy; otherwise the source's owner packs the source's state once per destination
    rank (sources in increasing id order), one all-to-all moves the packed states, and the receiver unpacks the slot of each
    of its destinations."""
    check_pairs(pairs, n_agents)
    own = _owner(n_agents, world)
    base = [shard_agents(n_agents, world, r).start for r in range(world)]
    routes = [RankRoute([], [], [], [], [0] * world, [0] * world, [], [], []) for _ in range(world)]
    sent: List[List[List[int]]] = [[[] for _ in range(world)] for _ in range(world)]       # sent[q][r]: sources q sends r
    for i, (s, d) in enumerate(pairs):
        rs, rd = own[s], own[d]
        if rs == rd:
            rt = routes[rs]
            rt.copy_src.append(s - base[rs]); rt.copy_dst.append(d - base[rs]); rt.copy_pair.append(i)
        elif s not in sent[rs][rd]:
            sent[rs][rd].append(s)
    for q in range(world):
        for r in range(world):
            sent[q][r].sort()
            routes[q].pack += [g - base[q] for g in sent[q][r]]
            routes[q].send_counts[r] = len(sent[q][r])
            routes[r].recv_counts[q] = len(sent[q][r])
    for i, (s, d) in enumerate(pairs):
        rs, rd = own[s], own[d]
        if rs != rd:
            slot = sum(len(sent[q][rd]) for q in range(rs)) + sent[rs][rd].index(s)
            rt = routes[rd]
            rt.unpack_slot.append(slot); rt.unpack_dst.append(d - base[rd]); rt.unpack_pair.append(i)
    return routes
