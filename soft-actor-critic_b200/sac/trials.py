"""Hyper-parameter trials as ONE population (SURVEY section 8f-2).

The reference's Optuna driver (hparam_search/scripts/run_search.py) materialises every trial as a YAML file and runs
``python main.py --config <trial.yaml>`` as a sequential subprocess (:58-65), scraping ``Final average return:`` from its stdout
(:74-80). Here the trials of a study become the agents of a ``SACPopulation``: every trial has its own environment instance,
replay ring, networks, optimiser state and device RNG streams, and every environment step of the study costs one batched
policy launch (``act_all``) plus -- once the rings are warm -- ONE update launch for all trials.

What may differ between trials are the scalars of the YAML's ``sac`` section (``SACPopulation.TRIAL_KEYS``: alpha, alpha_lr,
actor_lr, critic_lr, tau, gamma -- the shipped search space, hparam_search/configs/search_space.yaml, uses the first two);
anything that changes shapes (hidden sizes, batch size) has to be the same for the whole population and raises otherwise.
The search space file format and the ``section.param`` naming are the reference driver's (run_search.py:24-39).
"""
from __future__ import annotations

import copy
import math
import random as _random
from collections import deque
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .pbt import PBTConfig, explore, round_rng, select_pairs
from .population import SACPopulation, _dist


def sample_search_space(search_space: Dict[str, Dict[str, dict]], n_trials: int, seed: int = 0) -> List[Dict[str, Any]]:
    """n_trials draws from a run_search.py-style search space ({section: {param: {type, low/high | choices}}}); keys of the
    result are ``section.param`` as in ``trial.suggest_*`` (run_search.py:27-38). Independent sampling (what Optuna's default
    sampler does during its start-up trials); pass your own list of dicts to ``PopulationTrials`` to use another sampler."""
    rng = _random.Random(seed)
    out = []
    for _ in range(n_trials):
        t = {}
        for section, params in search_space.items():
            for param, st in params.items():
                if st["type"] == "categorical":
                    t[f"{section}.{param}"] = rng.choice(st["choices"])
                elif st["type"] == "uniform":
                    t[f"{section}.{param}"] = rng.uniform(st["low"], st["high"])
                elif st["type"] == "loguniform":
                    t[f"{section}.{param}"] = math.exp(rng.uniform(math.log(st["low"]), math.log(st["high"])))
                else:
                    raise ValueError(f"unknown search-space type {st['type']!r}")
        out.append(t)
    return out


def trial_config(base_config: dict, params: Dict[str, Any]) -> dict:
    """The YAML the reference driver would have written for this trial (run_search.py:18-39)."""
    cfg = copy.deepcopy(base_config)
    for key, value in params.items():
        section, param = key.split(".", 1)
        cfg.setdefault(section, {})[param] = value
    return cfg


class PopulationTrials:
    def __init__(self, base_config: dict, trials: Sequence[Dict[str, Any]], env_factory: Callable[[], Any], device=None,
                 rank: Optional[int] = None, world: Optional[int] = None,
                 search_space: Optional[Dict[str, Dict[str, dict]]] = None):
        """search_space (run_search.py format) bounds and redraws the values population-based training explores."""
        self.base_config = base_config
        self.search_space = search_space
        self.trials = [dict(t) for t in trials]
        self.lineage: List[List[Tuple[int, int, Dict[str, Any]]]] = [[] for _ in self.trials]     # (step, source, values)
        per_agent = []
        for i, t in enumerate(self.trials):
            pa = {}
            for key, value in t.items():
                section, param = key.split(".", 1)
                if section == "sac" and param in SACPopulation.TRIAL_KEYS:
                    pa[param] = float(value)
                elif trial_config(base_config, {key: value}) != base_config:
                    raise ValueError(f"trial {i}: {key} changes the population's structure; only sac.{{{', '.join(SACPopulation.TRIAL_KEYS)}}} "
                                     "may differ between the trials of one population")
            per_agent.append(pa)
        env0 = env_factory()
        obs_dim, act_dim = env0.observation_space.shape[0], env0.action_space.shape[0]
        seed = int(base_config["train"]["seed"])
        self.pop = SACPopulation(obs_dim, act_dim, base_config, len(self.trials), seeds=[seed + i for i in range(len(self.trials))],
                                 device=device, rank=rank, world=world)
        self.pop.set_trials(per_agent)
        self.envs = [env0] + [env_factory() for _ in range(self.pop.n_local - 1)]
        for a, env in enumerate(self.envs):                                     # SAC._set_seed per trial (agent.py:117-124)
            s = self.pop.seeds[a]
            env.reset(seed=s)
            env.action_space.seed(s)
            env.observation_space.seed(s)

    def run(self, num_episodes: int, out: Callable[[str], None] = print, pbt: Optional[PBTConfig] = None) -> List[Dict[str, float]]:
        """run_training_loop (agent.py:329-418) for every trial in lockstep: one environment step per trial per iteration, one
        update launch for all trials once every ring holds train.warming_steps transitions. Prints, per trial, the lines the
        reference driver prints / scrapes; returns the per-trial metrics dicts (total_episodes, best_avg_return,
        final_avg_return) in global trial order for this rank's trials.

        With a PBTConfig, population-based training: every pbt.interval_steps environment steps one exploit round (see
        sac/pbt.py) on the mean return of each trial's episodes since its last exploit (at most the last 100). A receiver
        takes its source's learner state and explored values (trial dict and lineage updated, return window emptied) and
        continues its environment episode; one line per pair: ``PBT step {t}: trial {dst} <- trial {src} {params}``."""
        pop, tr = self.pop, self.base_config["train"]
        n = pop.n_local
        update_every, grad_steps = tr.get("update_frequency", 1), tr.get("gradient_steps_per_update", 1)
        warming = tr["warming_steps"]
        states = [env.reset()[0] for env in self.envs]
        ep_ret, ep_done = [0.0] * n, [0] * n
        window = [deque(maxlen=100) for _ in range(n)]
        best = [-float("inf")] * n
        final: List[Optional[Dict[str, float]]] = [None] * n
        total_steps = 0
        obs_dim = pop.obs_dim
        rounds = 0
        # with ranks, finishing is decided at the exploit rounds (all ranks agree there), so every rank joins every round
        lockstep = pbt is not None and pop.world > 1
        running = True
        while running if lockstep else any(f is None for f in final):
            actions = pop.act_all(np.asarray(states, np.float32).reshape(n, obs_dim)).cpu().numpy()       # one launch, one D2H
            for a, env in enumerate(self.envs):
                if final[a] is not None:
                    continue
                nxt, reward, terminated, truncated, _ = env.step(actions[a])
                done = terminated or truncated
                pop.push(a, states[a], actions[a], reward, nxt, done)
                states[a] = nxt
                ep_ret[a] += reward
                if done:
                    window[a].append(ep_ret[a])
                    avg = float(np.mean(window[a]))
                    best[a] = max(best[a], avg)
                    ep_done[a] += 1
                    ep_ret[a] = 0.0
                    states[a] = env.reset()[0]
                    if ep_done[a] >= num_episodes:
                        g = pop.agent_ids[a]
                        final[a] = {"total_episodes": ep_done[a], "best_avg_return": best[a], "final_avg_return": avg}
                        out(f"--- Trial {g} Finished ---")
                        out(f"Trial {g} parameters: {self.trials[g]}")
                        out(f"Final average return: {avg}")
            total_steps += 1
            if total_steps >= warming and total_steps % update_every == 0:
                pop.update(grad_steps)
            if pbt is not None and total_steps % pbt.interval_steps == 0:
                local = [float(np.mean(window[a])) if final[a] is None and len(window[a]) >= pbt.min_episodes else None
                         for a in range(n)]
                scores, running = self._gather_scores(local, [f is None for f in final])
                rng = round_rng(pbt.seed, rounds)
                pairs = select_pairs(scores, pbt.fraction, rng)
                rounds += 1
                if pairs:
                    values = [explore(self.trials[s], self.search_space, pbt, rng) for s, _ in pairs]
                    pop.exploit(pairs, [{k.split(".", 1)[1]: v for k, v in vals.items()} for vals in values])
                    for (s, d), vals in zip(pairs, values):
                        self.trials[d] = vals
                        self.lineage[d].append((total_steps, s, dict(vals)))
                        if d in pop.agent_ids:
                            window[pop.local_index(d)].clear()
                        out(f"PBT step {total_steps}: trial {d} <- trial {s} {vals}")
        torch.cuda.synchronize()
        return [f for f in final if f is not None]

    def _gather_scores(self, local: List[Optional[float]], unfinished: List[bool]) -> Tuple[List[Optional[float]], bool]:
        """Every rank's scores in global trial order, and whether any trial anywhere is unfinished."""
        pop = self.pop
        d = _dist()
        if d is None or pop.world == 1:
            return list(local), any(unfinished)
        parts: List[Any] = [None] * pop.world
        d.all_gather_object(parts, (list(pop.agent_ids), list(local), any(unfinished)))
        scores: List[Optional[float]] = [None] * pop.n_agents_global
        for ids, vals, _ in parts:
            for g, v in zip(ids, vals):
                scores[g] = v
        return scores, any(p[2] for p in parts)


def run_population_search(base_config: dict, search_space: Dict[str, Dict[str, dict]], n_trials: int,
                          env_factory: Callable[[], Any], num_episodes: Optional[int] = None, seed: int = 0,
                          out: Callable[[str], None] = print) -> Dict[str, Any]:
    """The study of run_search.py (:151-176) as one population: sample n_trials configurations, train them concurrently, report
    the best -- same printed summary."""
    trials = sample_search_space(search_space, n_trials, seed)
    runner = PopulationTrials(base_config, trials, env_factory)
    metrics = runner.run(num_episodes or base_config["train"].get("num_episodes", 1000), out=out)
    values = [m["final_avg_return"] for m in metrics]
    best = int(np.argmax(values))
    out("\n\n--- Hyperparameter Search Finished ---")
    out(f"Number of finished trials: {len(values)}")
    out("\n--- Best Trial ---")
    out(f"  Trial Number: {best}")
    out(f"  Value (Final Avg Return): {values[best]:.4f}")
    out("\n  Best Hyperparameters:")
    for k, v in trials[best].items():
        out(f"    {k}: {v}")
    return {"trials": trials, "metrics": metrics, "best_trial": best, "best_value": values[best]}


def run_population_pbt(base_config: dict, search_space: Dict[str, Dict[str, dict]], n_trials: int, env_factory: Callable[[], Any],
                       pbt: PBTConfig, num_episodes: Optional[int] = None, seed: int = 0,
                       out: Callable[[str], None] = print) -> Dict[str, Any]:
    """run_population_search with population-based training: the same initial draws and printed summary; the best trial's
    "Best Hyperparameters" are the values in force at its end, followed by every trial's lineage."""
    trials = sample_search_space(search_space, n_trials, seed)
    runner = PopulationTrials(base_config, trials, env_factory, search_space=search_space)
    metrics = runner.run(num_episodes or base_config["train"].get("num_episodes", 1000), out=out, pbt=pbt)
    values = [m["final_avg_return"] for m in metrics]
    best = int(np.argmax(values))
    out("\n\n--- Hyperparameter Search Finished ---")
    out(f"Number of finished trials: {len(values)}")
    out("\n--- Best Trial ---")
    out(f"  Trial Number: {best}")
    out(f"  Value (Final Avg Return): {values[best]:.4f}")
    out("\n  Best Hyperparameters:")
    for k, v in runner.trials[best].items():
        out(f"    {k}: {v}")
    out("\n--- PBT Lineage ---")
    for g, steps in enumerate(runner.lineage):
        out(f"  Trial {g}: " + ("; ".join(f"step {t} <- trial {s} {vals}" for t, s, vals in steps) if steps else "initial values"))
    return {"trials": trials, "final_trials": runner.trials, "lineage": runner.lineage, "metrics": metrics, "best_trial": best,
            "best_value": values[best]}
