"""Multi-agent / multi-GPU modes of the update engine (SURVEY section 8e). Neither exists in the reference:
its only "parallelism" is the Optuna driver launching sequential ``main.py`` subprocesses
(hparam_search/scripts/run_search.py:58-65,151-155).

``SACPopulation``     independent agents (seeds / trials): each has private parameters, Adam state, targets,
                      temperature, replay ring and RNG streams. Agents are partitioned over ranks in contiguous
                      blocks and updated by ONE launch per rank (one CTA per agent, agents looped per CTA);
                      there is NO collective on the data path -- only an optional gather of scalar metrics.
``DataParallelSAC``   one agent, global batch split B/G rows per rank, parameters replicated. The critic step
                      precedes the actor forward (F4), so there are two exchange points per update:
                      all-reduce(sum) of the critic gradients, then ONE all-reduce of the policy gradients with the
                      temperature-gradient share stored right behind them. NCCL over NVLink through torch.distributed, on the engine's stream.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _engine as E
from .engine import UpdateEngine
from .models import PolicyNetwork, QNetwork
from .replay_buffer import ReplayBuffer


def shard_agents(n_agents: int, world: int, rank: int) -> range:
    """Contiguous block of global agent ids owned by `rank` (sizes differ by at most one)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, extra = divmod(n_agents, world)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def split_batch(global_batch: int, world: int) -> int:
    """Rows per rank of a data-parallel batch; equal shards keep the mean-loss semantics exact."""
    if global_batch % world:
        raise ValueError(f"global batch {global_batch} is not divisible by the number of ranks {world}")
    return global_batch // world


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


class SACPopulation:
    def __init__(self, obs_dim: int, act_dim: int, config: dict, n_agents: int, seeds: Optional[Sequence[int]] = None,
                 device=None, rank: Optional[int] = None, world: Optional[int] = None, reference_init: bool = True):
        if E.per_config(config) is not None:
            raise ValueError("buffer.prioritized is not supported by SACPopulation")
        d = _dist()
        self.world = world if world is not None else (d.get_world_size() if d else 1)
        self.rank = rank if rank is not None else (d.get_rank() if d else 0)
        self.n_agents_global = int(n_agents)
        self.agent_ids = list(shard_agents(n_agents, self.world, self.rank))
        self.n_local = len(self.agent_ids)
        if self.n_local == 0:
            raise ValueError("more ranks than agents")
        self.seeds = [int(seeds[g]) if seeds is not None else g for g in self.agent_ids]
        self.config = config
        self.obs_dim, self.act_dim = obs_dim, act_dim
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        # device RNG streams (replay indices, policy noise, rollout noise) are keyed by (seed, GLOBAL agent id): two ranks'
        # local agent 0 draw different streams; an agent's own seed (seeds[g]) replaces train.seed as its first key
        self.engine = UpdateEngine(obs_dim, act_dim, config, device=dev, n_agents=self.n_local, agent_id_base=self.agent_ids[0])
        self.ring = ReplayBuffer(config["buffer"]["capacity"], obs_dim, act_dim, device=dev, n_agents=self.n_local)
        self._init_weights(reference_init)
        self.engine.reset_state()
        if seeds is not None:
            for a, seed in enumerate(self.seeds):
                self.engine.view("scal.rng_seed", a).fill_(int(seed))
        self.engine.attach_ring(self.ring)

    def _init_weights(self, reference_init: bool) -> None:
        pn, qn = self.config["policy_net"], self.config["q_net"]
        eng = self.engine
        if reference_init:
            # per agent: the reference's constructor calls with that agent's seed (policy/Q1: seed, Q2: seed+1)
            for a, seed in enumerate(self.seeds):
                nets = {
                    "pi": PolicyNetwork(self.obs_dim, self.act_dim, pn["hidden_sizes"], hidden_activations=pn["hidden_layers_act"],
                                        output_activation=pn["output_activation"], seed=seed),
                    "q1": QNetwork(self.obs_dim, self.act_dim, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed),
                    "q2": QNetwork(self.obs_dim, self.act_dim, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed + 1),
                }
                for tag, net in nets.items():
                    for l, lin in enumerate(net.linears()):
                        eng.view(f"{tag}.W{l}", a).copy_(lin.weight.detach())
                        eng.view(f"{tag}.b{l}", a).reshape(-1).copy_(lin.bias.detach())
        else:
            # fast path for large populations: xavier_uniform_ drawn on the device, one stream per rank
            g = torch.Generator(device=eng.device).manual_seed(1234 + self.agent_ids[0])
            for tag, n_lin in (("pi", len(pn["hidden_sizes"]) + 1), ("q1", len(qn["hidden_sizes"]) + 1), ("q2", len(qn["hidden_sizes"]) + 1)):
                for l in range(n_lin):
                    v = eng.population_view(f"{tag}.W{l}")
                    bound = (6.0 / (v.shape[1] + v.shape[2])) ** 0.5
                    v.copy_((torch.rand(v.shape, device=eng.device, generator=g) * 2 - 1) * bound)

    # ------------------------------------------------------------------ data
    def local_index(self, global_agent: int) -> int:
        return self.agent_ids.index(global_agent)

    def push(self, agent: int, state, action, reward, next_state, done) -> None:
        self.ring.push(state, action, reward, next_state, done, agent=agent)

    def push_batch(self, agent: int, s, a, r, s2, d) -> None:
        self.ring.push_batch(s, a, r, s2, d, agent=agent)

    def push_device_all(self, s, a, r, s2, d) -> None:
        """Same device-resident rows into every local agent's ring (synthetic benchmarks)."""
        for ag in range(self.n_local):
            self.ring.push_device(s, a, r, s2, d, agent=ag)

    # ------------------------------------------------------------------ compute
    def update(self, n_steps: int = 1) -> None:
        """n_steps updates of every local agent: one kernel launch, no collective."""
        self.engine.update(None, None, None, n_steps)

    # ------------------------------------------------------------------ trials (SURVEY 8f-2)
    # hyper-parameters the engine keeps PER AGENT (scalar block of the arena): every scalar of the YAML's `sac` section
    TRIAL_KEYS = ("alpha", "alpha_lr", "actor_lr", "critic_lr", "tau", "gamma")

    def set_trial(self, agent: int, alpha: Optional[float] = None, alpha_lr: Optional[float] = None,
                  actor_lr: Optional[float] = None, critic_lr: Optional[float] = None, tau: Optional[float] = None,
                  gamma: Optional[float] = None) -> None:
        """Per-agent values of the `sac.*` scalars for local agent `agent` (one Optuna trial per agent; the reference's driver
        is generic over any section/param: hparam_search/scripts/run_search.py:24-39; its shipped search space uses
        ``sac.alpha`` and ``sac.alpha_lr``: hparam_search/configs/search_space.yaml). Same roundings as the reference applies
        to the config values: learning rates stay python doubles (torch.optim.Adam), gamma / tau / 1 - tau become float32
        scalars (agent.py:208,288-291), log_alpha = log(alpha) in float64 (agent.py:45-50). Call before the first update."""
        import math
        eng = self.engine
        eng.sync()
        if alpha is not None:
            if not alpha > 0:
                raise ValueError("alpha must be positive")
            la = math.log(alpha)          # agent.py:49-50: log_alpha = log(alpha) in float64, alpha = exp(log_alpha)
            eng.view("scal.log_alpha", agent).fill_(la)
            eng.view("scal.alpha", agent).fill_(math.exp(la) if self.config["sac"]["auto_entropy_tuning"] else float(np.float32(alpha)))
        if alpha_lr is not None:
            if not alpha_lr > 0:
                raise ValueError("alpha_lr must be positive")
            eng.view("scal.alpha_lr", agent).fill_(float(alpha_lr))
        lr = eng.view("scal.lr", agent)
        if actor_lr is not None:
            if not actor_lr > 0:
                raise ValueError("actor_lr must be positive")
            lr[0] = float(actor_lr)
        if critic_lr is not None:
            if not critic_lr > 0:
                raise ValueError("critic_lr must be positive")
            lr[1] = float(critic_lr)
            lr[2] = float(critic_lr)
        if tau is not None:
            if not 0.0 <= tau <= 1.0:
                raise ValueError("tau must be in [0, 1]")
            t = eng.view("scal.tau", agent).reshape(-1)
            t[0] = float(np.float32(tau))
            t[1] = float(np.float32(1.0 - tau))      # the python double 1.0 - tau rounded once, as in agent.py:290
        if gamma is not None:
            eng.view("scal.gamma", agent).fill_(float(np.float32(gamma)))
        eng.refresh_alpha()

    def set_trials(self, trials: Sequence[Dict[str, float]]) -> None:
        """trials[g] = {"alpha": ..., "alpha_lr": ..., "actor_lr": ..., "critic_lr": ..., "tau": ..., "gamma": ...} (any subset)
        for GLOBAL agent g (one Optuna trial per agent); this rank applies its own block. The sequential `subprocess.run` loop
        of hparam_search/scripts/run_search.py:58-65 becomes one population."""
        if len(trials) != self.n_agents_global:
            raise ValueError("one trial per agent expected")
        for a, g in enumerate(self.agent_ids):
            unknown = set(trials[g]) - set(self.TRIAL_KEYS)
            if unknown:
                raise KeyError(f"not a per-agent hyper-parameter: {sorted(unknown)} (per-agent: {self.TRIAL_KEYS})")
            self.set_trial(a, **{k: trials[g].get(k) for k in self.TRIAL_KEYS})

    def exploit(self, pairs: Sequence[Tuple[int, int]], hypers: Optional[Sequence[Optional[Dict[str, float]]]] = None) -> None:
        """Population-based training's exploit (and explore) step: for every (source, destination) pair of GLOBAL agent ids the
        destination takes over the source's learner state -- parameters, Adam state, targets, temperature and its optimiser,
        step counters and hyper-parameters -- and keeps its own replay ring, update counter, RNG streams and metrics; then
        hypers[i] (a dict over a subset of TRIAL_KEYS, or None) is written into pair i's destination with set_trial's
        roundings. Every copy reads the state from before the call: a destination may not be a source, a source may feed
        several destinations. Like set_trials, every rank calls it with the same arguments. Pairs within a rank are one
        launch; pairs across ranks add a pack launch, ONE all_to_all_single on the engine's stream, and an unpack launch. The
        result does not depend on the sharding."""
        from .pbt import pbt_record, route_exploit
        pairs = [(int(s), int(d)) for s, d in pairs]
        if hypers is not None and len(hypers) != len(pairs):
            raise ValueError("one hyper-parameter dict (or None) per pair expected")
        routes = route_exploit(pairs, self.n_agents_global, self.world)
        rt = routes[self.rank]
        records = None
        if hypers is not None:
            auto = bool(self.config["sac"]["auto_entropy_tuning"])
            records = [pbt_record(h, auto) for h in hypers]
        eng = self.engine
        if rt.copy_dst:
            eng.pbt_copy(rt.copy_src, rt.copy_dst, None if records is None else [records[i] for i in rt.copy_pair])
        if not any(r.pack for r in routes):
            return
        d = _dist()
        if d is None or d.get_world_size() != self.world:
            raise RuntimeError("exploit: pairs across ranks need the torch.distributed process group the population is sharded over")
        F = eng.pbt_state_floats()
        send = torch.empty((len(rt.pack), F), dtype=torch.float32, device=eng.device)
        recv = torch.empty((sum(rt.recv_counts), F), dtype=torch.float32, device=eng.device)
        eng.pbt_pack(rt.pack, send)
        d.all_to_all_single(recv, send, output_split_sizes=rt.recv_counts, input_split_sizes=rt.send_counts)
        eng.pbt_unpack(recv, rt.unpack_slot, rt.unpack_dst, None if records is None else [records[i] for i in rt.unpack_pair])

    def act_all(self, states, deterministic: bool = False, eps=None) -> torch.Tensor:
        """One action per local agent from its own observation (vectorised envs): states [n_local, obs] (numpy or tensor) ->
        device tensor [n_local, act]; one kernel launch for the whole population (reference: select_action per agent,
        agent.py:149-156)."""
        s = torch.as_tensor(np.asarray(states, np.float32) if not torch.is_tensor(states) else states)
        return self.engine.act_population(s.view(self.n_local, 1, self.obs_dim), eps, deterministic)[:, 0, :]

    def act(self, agent: int, state, deterministic: bool = False) -> np.ndarray:
        return self.engine.act_host(np.asarray(state, np.float32), None, deterministic, agent=agent)[0]

    def metrics(self, agent: int) -> dict:
        return self.engine.metrics(agent)

    def gather_metrics(self, key: str = "q1_loss") -> Optional[np.ndarray]:
        """Host-side gather of one scalar per agent onto rank 0 (the only cross-rank traffic of this mode)."""
        vals = torch.tensor([self.engine.metrics(a)[key] for a in range(self.n_local)], dtype=torch.float64)
        d = _dist()
        if d is None or self.world == 1:
            return vals.numpy()
        sizes = [len(shard_agents(self.n_agents_global, self.world, r)) for r in range(self.world)]
        pad = torch.zeros(max(sizes), dtype=torch.float64)
        pad[: self.n_local] = vals
        buf = pad.cuda() if d.get_backend() == "nccl" else pad
        out = [torch.zeros_like(buf) for _ in range(self.world)]
        d.all_gather(out, buf)
        if self.rank != 0:
            return None
        return np.concatenate([o.cpu().numpy()[:n] for o, n in zip(out, sizes)])

    def agent_state_dict(self, agent: int) -> Dict[str, Dict[str, torch.Tensor]]:
        """Reference-schema network state_dicts of one local agent (checkpoint interchange, agent.py:521-536)."""
        out = {}
        for key, tag in (("policy_net_state_dict", "pi"), ("q_net1_state_dict", "q1"), ("q_net2_state_dict", "q2"),
                         ("q_net1_target_state_dict", "q1t"), ("q_net2_target_state_dict", "q2t")):
            n_lin = len(self.config["policy_net" if tag == "pi" else "q_net"]["hidden_sizes"]) + 1
            sd = {}
            for l in range(n_lin):
                sd[f"net.{2 * l}.weight"] = self.engine.view(f"{tag}.W{l}", agent).detach().clone()
                sd[f"net.{2 * l}.bias"] = self.engine.view(f"{tag}.b{l}", agent).reshape(-1).detach().clone()
            out[key] = sd
        return out


class DataParallelSAC:
    """Large-batch data-parallel SAC (BASELINE config 5): global batch B, B/G rows per rank, ring replicated."""

    def __init__(self, obs_dim: int, act_dim: int, config: dict, global_batch: int, device=None,
                 rank: Optional[int] = None, world: Optional[int] = None):
        if E.per_config(config) is not None:
            raise ValueError("buffer.prioritized is not supported by DataParallelSAC")
        d = _dist()
        self.world = world if world is not None else (d.get_world_size() if d else 1)
        self.rank = rank if rank is not None else (d.get_rank() if d else 0)
        self.local_batch = split_batch(global_batch, self.world)
        self.global_batch = global_batch
        self.config, self.obs_dim, self.act_dim = config, obs_dim, act_dim
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.engine = UpdateEngine(obs_dim, act_dim, config, device=dev, dp_world=self.world, dp_rank=self.rank,
                                   batch_size=self.local_batch)
        self.ring = ReplayBuffer(config["buffer"]["capacity"], obs_dim, act_dim, device=dev)
        pn, qn, seed = config["policy_net"], config["q_net"], config["train"]["seed"]
        nets = {
            "pi": PolicyNetwork(obs_dim, act_dim, pn["hidden_sizes"], hidden_activations=pn["hidden_layers_act"],
                                output_activation=pn["output_activation"], seed=seed),
            "q1": QNetwork(obs_dim, act_dim, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed),
            "q2": QNetwork(obs_dim, act_dim, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed + 1),
        }
        for tag, net in nets.items():              # identical on every rank (same seed)
            for l, lin in enumerate(net.linears()):
                self.engine.view(f"{tag}.W{l}").copy_(lin.weight.detach())
                self.engine.view(f"{tag}.b{l}").reshape(-1).copy_(lin.bias.detach())
        self.engine.reset_state()
        self.engine.attach_ring(self.ring)
        self.g_critics = self.engine.view("block.g.critics").reshape(-1)
        # exchange #2 is ONE message: the policy gradients with this rank's temperature-gradient share right behind them
        self.g_policy = self.engine.view("block.g.policy_x").reshape(-1)
        self.time_exchange = False            # bench: CUDA events around the two exchanges
        self._events = []

    def _allreduce(self, t: torch.Tensor) -> None:
        d = _dist()
        if d is not None and self.world > 1:
            if self.time_exchange:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                d.all_reduce(t, op=d.ReduceOp.SUM)
                e1.record()
                self._events.append((e0, e1))
            else:
                d.all_reduce(t, op=d.ReduceOp.SUM)

    def exchange_ms(self) -> float:
        """Device time spent inside the all-reduces since the last call (needs time_exchange = True; synchronises)."""
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in self._events)
        self._events = []
        return ms

    # The update in three local segments separated by the two exchange points (F4).
    def segment_critic_grads(self, idx=None, eps1=None) -> None:
        e = self.engine
        e.sample_batch(idx)
        e.target(eps1)
        e.critic_step(None, grads_only=True)          # gradients carry the 1/B_global factor

    def segment_critic_apply_actor_grads(self, eps2=None) -> None:
        e = self.engine
        e.apply_grads(1, polyak=True)                 # Adam on Q1, Q2 + Polyak (critics do not change afterwards)
        e.actor_step(eps2, None, grads_only=True)

    def segment_actor_apply(self) -> None:
        self.engine.apply_grads(2 | 4)                # Adam on the policy, temperature step, update counter

    def update(self, idx: Optional[torch.Tensor] = None, eps1: Optional[torch.Tensor] = None,
               eps2: Optional[torch.Tensor] = None) -> None:
        """One global-batch update. idx/eps (device tensors) hold THIS rank's rows; None = device RNG keyed by
        the global row id, so the global batch is the same for every G."""
        self.segment_critic_grads(idx, eps1)
        self._allreduce(self.g_critics)               # exchange #1: 588 KB at BipedalWalker shape
        self.segment_critic_apply_actor_grads(eps2)
        self._allreduce(self.g_policy)                # exchange #2: 297 KB, the temperature-gradient share rides along
        self.segment_actor_apply()
