"""``SAC``: the reference agent's class surface on top of the B200 update engine.

Reference: /root/reference/sac/agent.py.  Method-by-method correspondence (file:line of the
reference method each one replaces) is given in the docstrings; INTEGRATION.md has the table.

What is different underneath:
  * one gradient update (``training_step``, agent.py:302-327) is ONE launch of the persistent fused
    CUDA kernel (``sacx_update``): ring gather -> soft Bellman target -> twin-critic forward/backward
    with Adam and the Polyak update in the dW epilogue -> actor forward/backward with Adam ->
    temperature step.  Nothing of it runs in PyTorch.
  * networks, targets, Adam moments and ``log_alpha`` live in one packed device arena; the
    ``nn.Module`` / optimiser / ``log_alpha`` attributes are zero-copy views of it, so
    ``state_dict()``, ``load_state_dict()`` and the checkpoint schema (agent.py:521-554) are unchanged.
  * ``train.device`` must be a CUDA device.  There is no CPU fallback for the update path.

Optional config keys (all default so that every reference YAML loads unchanged):
  ``train.rng``: ``"device"`` (default; Feistel index sampling + Philox normals inside the kernel) or
  ``"host"`` (reference streams: indices from Python's global ``random``, normals from torch's CPU
  generator -- bit-identical index stream, used by the parity tests and the e2e benchmark).
  ``buffer.prioritized``: ``{alpha: 0.6, beta: 0.4, beta_steps: 0, eps: 1e-6}`` (missing keys take these defaults) turns on
  prioritized experience replay on the device (``PrioritizedReplayBuffer``; single agent, ``train.rng: device``); absent or
  null keeps uniform sampling.
"""
from __future__ import annotations

import copy
import os
import pprint
import random
from collections import deque
from typing import Any, Dict, Optional

import numpy as np
import torch
import torch.optim as optim

from . import _engine as E
from .engine import UpdateEngine
from .models import PolicyNetwork, QNetwork
from .replay_buffer import PrioritizedReplayBuffer, ReplayBuffer, Transition

try:  # progress bars are optional plumbing
    from tqdm import tqdm
except Exception:  # pragma: no cover
    def tqdm(it, disable=False):
        return it


class _EngineAdam(optim.Adam):
    """``torch.optim.Adam`` facade over moments that the CUDA kernels own.

    ``state_dict()`` / ``load_state_dict()`` keep torch's schema (what the reference checkpoints
    hold, agent.py:529-535); ``step()`` is refused -- the fused update applies Adam itself."""

    def bind(self, engine: UpdateEngine, opt_index: int, moment_views) -> None:
        self._engine, self._opt_index = engine, opt_index
        self._moments = moment_views
        for p, (m, v) in zip(self.param_groups[0]["params"], moment_views):
            self.state[p] = {"step": torch.tensor(0.0), "exp_avg": m, "exp_avg_sq": v}

    def _device_step(self) -> int:
        return int(self._engine.view("scal.step")[self._opt_index].item())

    def state_dict(self):
        t = float(self._device_step())
        for p in self.param_groups[0]["params"]:
            self.state[p]["step"] = torch.tensor(t)
        return super().state_dict()

    def load_state_dict(self, state_dict) -> None:
        """torch.optim.Adam.load_state_dict semantics on engine-owned moments: the moments and the step counter go into the
        arena, the checkpoint's param_groups (lr, betas, eps, ...) replace this optimiser's -- a checkpoint saved with another
        learning rate resumes with THAT rate, as it does in the reference -- and the rate is pushed into the engine."""
        st = state_dict.get("state", {})
        groups = state_dict.get("param_groups", [])
        if st and len(st) != len(self._moments):
            raise ValueError(f"loaded state dict has {len(st)} parameter states, this optimizer has {len(self._moments)}")
        if groups:
            if len(groups) != 1 or len(groups[0].get("params", [])) != len(self._moments):
                raise ValueError("loaded state dict contains a parameter group that doesn't match the size of optimizer's group")
            g = groups[0]
            if tuple(g.get("betas", (0.9, 0.999))) != (0.9, 0.999) or g.get("eps", 1e-8) != 1e-8 or g.get("weight_decay", 0) != 0 \
                    or g.get("amsgrad", False) or g.get("maximize", False):
                raise ValueError("the fused update implements torch.optim.Adam's defaults only (betas (0.9, 0.999), eps 1e-8, "
                                 "no weight decay / amsgrad / maximize): this checkpoint's optimiser uses something else")
        step = None
        with torch.no_grad():
            for i, (m, v) in enumerate(self._moments):
                ent = st.get(i, st.get(str(i)))
                if ent is None:
                    m.zero_()
                    v.zero_()
                    continue
                ea, es = torch.as_tensor(ent["exp_avg"]), torch.as_tensor(ent["exp_avg_sq"])
                if ea.numel() != m.numel() or es.numel() != v.numel():
                    raise ValueError(f"optimizer state {i}: shape {tuple(ea.shape)} does not match the parameter's {tuple(m.shape)}")
                m.copy_(ea.to(m.device).reshape(m.shape))
                v.copy_(es.to(v.device).reshape(v.shape))
                s_i = int(float(ent["step"]))
                if step is not None and s_i != step:
                    raise ValueError("per-parameter Adam step counters differ: the fused update keeps one counter per optimiser")
                step = s_i
            self._engine.view("scal.step")[self._opt_index] = step or 0
            if groups:
                lr = float(groups[0]["lr"])
                for k, val in groups[0].items():
                    if k != "params":
                        self.param_groups[0][k] = val
                if self._opt_index < 3:
                    self._engine.view("scal.lr")[self._opt_index] = lr
                else:
                    cur = float(self._engine.view("scal.alpha_lr").item())
                    self._engine.view("scal.alpha_lr").fill_(-abs(lr) if cur < 0 else lr)

    def step(self, closure=None):
        raise RuntimeError("parameters are stepped by the fused CUDA update (SAC.training_step), not by torch")


class SAC:
    def __init__(self, env, config: dict):
        """reference: agent.py:22-67 (+ _init_policy_network / _init_q_networks / _init_optimizers / _set_seed)."""
        self.env = env
        self.config = config
        self.device = torch.device(config["train"]["device"])
        if self.device.type != "cuda":
            raise RuntimeError(
                f"train.device={config['train']['device']!r}: this SAC runs its update on a CUDA device "
                "(B200, sm_100a) and has no CPU fallback; set train.device to 'cuda'")
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device available for the SAC update engine")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.obs_size = env.observation_space.shape[0]
        self.action_size = env.action_space.shape[0]
        self.rng_mode = config["train"].get("rng", "device")
        if self.rng_mode not in ("device", "host"):
            raise ValueError("train.rng must be 'device' or 'host'")
        seed = config["train"]["seed"]
        pn, qn = config["policy_net"], config["q_net"]
        self.per = E.per_config(config)            # buffer.prioritized: None -> uniform sampling

        if self.per is None:
            self.replay_buffer = ReplayBuffer(config["buffer"]["capacity"], self.obs_size, self.action_size, device=self.device)
        else:
            self.replay_buffer = PrioritizedReplayBuffer(
                config["buffer"]["capacity"], self.obs_size, self.action_size, device=self.device, alpha=self.per["alpha"],
                beta=self.per["beta"], beta_steps=self.per["beta_steps"], eps=self.per["eps"],
                max_batch=config["train"]["batch_size"], seed=seed)

        # networks: same constructor calls and seeds as the reference (policy/Q1: seed, Q2: seed+1)
        self.policy_net = PolicyNetwork(self.obs_size, self.action_size, pn["hidden_sizes"], log_std_min=pn["log_std_min"],
                                        log_std_max=pn["log_std_max"], action_scale=pn["action_scale"],
                                        hidden_activations=pn["hidden_layers_act"], output_activation=pn["output_activation"], seed=seed)
        self.q_net1 = QNetwork(self.obs_size, self.action_size, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed)
        self.q_net2 = QNetwork(self.obs_size, self.action_size, qn["hidden_sizes"], qn["hidden_layers_act"], qn["output_activation"], seed=seed + 1)
        self.q_net1_target = copy.deepcopy(self.q_net1)
        self.q_net2_target = copy.deepcopy(self.q_net2)

        self.engine = UpdateEngine(self.obs_size, self.action_size, config, device=self.device)
        self.engine.attach_ring(self.replay_buffer)
        if self.per is not None:
            self.engine.attach_per(self.replay_buffer)
        views = self._views = self.engine.views()
        self.policy_net.bind_to_views(views, "pi")
        self.q_net1.bind_to_views(views, "q1")
        self.q_net2.bind_to_views(views, "q2")
        self.engine.reset_state()                      # targets <- critics, Adam state zero, temperature from config
        self.q_net1_target.bind_to_views(views, "q1t", copy_in=False)
        self.q_net2_target.bind_to_views(views, "q2t", copy_in=False)

        self.policy_optimizer = self._make_optimizer(self.policy_net, "pi", 0, config["sac"]["actor_lr"])
        self.q1_optimizer = self._make_optimizer(self.q_net1, "q1", 1, config["sac"]["critic_lr"])
        self.q2_optimizer = self._make_optimizer(self.q_net2, "q2", 2, config["sac"]["critic_lr"])

        self._set_seed(seed)

        self.target_entropy = -float(self.action_size)
        self.auto_entropy = bool(config["sac"]["auto_entropy_tuning"])
        if self.auto_entropy:
            self.log_alpha = views["scal.log_alpha"].reshape(())          # 0-dim float64, live
            self.alpha_optimizer = _EngineAdam([self.log_alpha], lr=config["sac"]["alpha_lr"])
            self.alpha_optimizer.bind(self.engine, 3, [(views["scal.alpha_m"].reshape(()), views["scal.alpha_v"].reshape(()))])
        else:
            self._fixed_alpha = torch.tensor(config["sac"]["alpha"]).to(self.device)

        lg = config["logger"]
        self.env_name = lg["env_name"] or self._infer_env_name(env)
        self.agent_name = lg["agent_name"] or self.__class__.__name__
        self.logger = None
        if lg["enabled"]:
            from .utils.experiment_logger import ExperimentLogger
            self.logger = ExperimentLogger(lg, env_name=self.env_name, agent_name=self.agent_name)

    # ------------------------------------------------------------------ construction helpers
    def _make_optimizer(self, net, tag: str, opt_index: int, lr: float) -> _EngineAdam:
        opt = _EngineAdam(net.parameters(), lr=lr)
        pairs = []
        for l, _ in enumerate(net.linears()):
            pairs.append((self._views[f"m.{tag}.W{l}"], self._views[f"v.{tag}.W{l}"]))
            pairs.append((self._views[f"m.{tag}.b{l}"].reshape(-1), self._views[f"v.{tag}.b{l}"].reshape(-1)))
        opt.bind(self.engine, opt_index, pairs)
        return opt

    def _set_seed(self, seed: int) -> None:
        """reference: agent.py:117-124."""
        np.random.seed(seed)
        torch.manual_seed(seed)
        random.seed(seed)
        self.env.reset(seed=seed)
        self.env.action_space.seed(seed)
        self.env.observation_space.seed(seed)

    @property
    def alpha(self) -> torch.Tensor:
        """Temperature: float64 0-dim (auto-tuned, exp(log_alpha)) or float32 0-dim (fixed) -- F6."""
        if self.auto_entropy:
            return self._views["scal.alpha"].reshape(())
        return self._fixed_alpha

    def _normal(self, rows: int) -> Optional[np.ndarray]:
        """The draw ``Normal.rsample`` makes on the reference's CPU path (models.py:82-83)."""
        if self.rng_mode != "host":
            return None
        return torch.empty(rows, self.action_size).normal_().numpy()

    def _normal_pair(self, rows: int):
        """The two consecutive draws of one update (pi(s'), then pi(s)). torch's CPU normal_ fills 16-element blocks
        independently (uniforms first, Box-Muller inside each block), so ONE draw of 2 x rows x A elements is the same stream as
        two draws of rows x A whenever rows x A is a multiple of 16 (tests/test_binding_cpu.py pins this); otherwise two draws."""
        n = rows * self.action_size
        if n % 16 == 0 and n >= 16:
            both = torch.empty(2, rows, self.action_size).normal_().numpy()
            return both[0], both[1]
        return self._normal(rows), self._normal(rows)

    # ------------------------------------------------------------------ buffer side
    def store_transition(self, state: Any, action: Any, reward: float, next_state: Any, done: bool) -> None:
        """reference: agent.py:126-135."""
        self.replay_buffer.push(state, action, reward, next_state, done)

    def warmup_replay_buffer(self, env: Any, steps: int) -> None:
        """reference: agent.py:137-147 -- prefill with uniformly random actions."""
        state, _ = env.reset()
        for _ in range(steps):
            action = env.action_space.sample()
            next_state, reward, terminated, truncated, _ = env.step(action)
            done = terminated or truncated
            self.store_transition(state, action, reward, next_state, done)
            state = env.reset()[0] if done else next_state

    def can_update(self) -> bool:
        """reference: agent.py:159-164."""
        if self.config["train"]["warming_steps"] > self.config["buffer"]["capacity"]:
            print("Warning: warming_steps is greater than replay buffer capacity.")
        return len(self.replay_buffer) >= self.config["train"]["warming_steps"]

    def sample_batch(self) -> Transition:
        """reference: agent.py:166-193 -- float32 device tensors for a ``random.sample`` index draw.

        With ``buffer.n_step`` > 1 the batch is gathered by the engine, so the per-phase methods see the folded batch
        ``training_step`` trains on (n-step return, next state at the window's end, encoded done column): indices from the
        reference's stream in host-RNG mode, else the device draw the next ``training_step`` would make."""
        B = self.config["train"]["batch_size"]
        if self.engine.cfg.n_step <= 1:
            return ReplayBuffer.sample_tensors(self.replay_buffer, B)
        idx = None
        if self.rng_mode == "host":
            idx = torch.as_tensor(np.asarray(self.replay_buffer.draw_indices(B), dtype=np.int64)).to(self.device)
        else:
            self.replay_buffer._require(B)
        self.engine.sample_batch(idx)
        sa, s2a, O = self._views["batch.sa"], self._views["batch.s2a"], self.obs_size
        return Transition(sa[:, :O].clone(), sa[:, O:].clone(), self._views["batch.r"].reshape(-1).clone(),
                          s2a[:, :O].clone(), self._views["batch.d"].reshape(-1).clone())

    # ------------------------------------------------------------------ acting
    def select_action(self, state: Any, deterministic: bool = False) -> Any:
        """reference: agent.py:149-156 (policy forward at batch 1 -> numpy action)."""
        eps = None if deterministic else self._normal(1)
        return self.engine.act_host(np.asarray(state, dtype=np.float32), eps, deterministic)[0]

    # ------------------------------------------------------------------ the update, phase by phase
    def _f32(self, t) -> torch.Tensor:
        return torch.as_tensor(t, dtype=torch.float32, device=self.device).contiguous()

    def _dev_normal(self) -> Optional[torch.Tensor]:
        e = self._normal(self.config["train"]["batch_size"])
        return None if e is None else torch.from_numpy(e).to(self.device)

    def compute_target_q_values(self, rewards: Any, dones: Any, next_states: Any) -> Any:
        """reference: agent.py:195-211 -- y = r + gamma (1-d) (min Q_target(s', a') - alpha log pi(a'|s'))."""
        self.engine.load_batch(s2=self._f32(next_states), r=self._f32(rewards), d=self._f32(dones))
        y = torch.empty(self.config["train"]["batch_size"], dtype=torch.float32, device=self.device)
        self.engine.target(self._dev_normal(), y)
        return y

    def update_q_networks(self, states: Any, actions: Any, target_q_values: Any) -> None:
        """reference: agent.py:213-236 -- twin-critic MSE step (Adam on Q1, then Q2)."""
        self.engine.load_batch(s=self._f32(states), a=self._f32(actions))
        self.engine.critic_step(self._f32(target_q_values))

    def update_policy_network(self, states: Any):
        """reference: agent.py:238-260 -- reparameterised actor step; returns log pi [B]."""
        self.engine.load_batch(s=self._f32(states))
        lp = torch.empty(self.config["train"]["batch_size"], dtype=torch.float32, device=self.device)
        self.engine.actor_step(self._dev_normal(), lp)
        return lp

    def update_entropy_temperature(self, log_pi: Any) -> Dict[str, float]:
        """reference: agent.py:263-280."""
        if not self.auto_entropy:
            return {}
        m = self.engine.alpha_step(self._f32(log_pi), want_metrics=True)
        return {"alpha_loss": m["alpha_loss"], "alpha": m["alpha"]}

    def soft_update_target_networks(self) -> None:
        """reference: agent.py:282-300."""
        self.engine.polyak()

    def training_step(self) -> None:
        """reference: agent.py:302-327 -- one full gradient update, one fused kernel launch.

        Host-RNG mode submits the update software-pipelined (H2D of this step's index stream + normals, kernel, D2H of the
        metrics block; the metrics of the PREVIOUS step are collected while this one runs), so the host draws step t+1 while
        step t executes. A non-finite policy head -- where the reference's ``Normal(mu, std)`` raises ValueError at once -- is
        reported here one step late, from the collected metrics."""
        B = self.config["train"]["batch_size"]
        if self.rng_mode == "host":
            idx = np.asarray(self.replay_buffer.draw_indices(B), dtype=np.int64)
            e1, e2 = self._normal_pair(B)
            m = self.engine.update_host_pipelined(idx, e1, e2, 1)
            self._host_pending = True
            if m is not None and m["nonfinite"]:
                raise ValueError("policy head produced non-finite mean/std (torch Normal would have rejected them)")
        else:
            if len(self.replay_buffer) < B:
                self.replay_buffer._require(B)
            self.engine.update(None, None, None, 1)

    def training_steps(self, n: int) -> None:
        """n consecutive updates inside one launch (device RNG); the UTD>1 burst of
        ``gradient_steps_per_update`` (agent.py:366-369) collapses to this."""
        if self.rng_mode == "host":
            for _ in range(n):
                self.training_step()
        else:
            self.replay_buffer._require(self.config["train"]["batch_size"])
            self.engine.update(None, None, None, int(n))

    def last_metrics(self) -> Dict[str, float]:
        """Device-side losses / temperature of the most recent update (synchronises)."""
        if getattr(self, "_host_pending", False):
            self.engine.update_host_flush()
            self._host_pending = False
        m = self.engine.metrics()
        if m["nonfinite"]:
            raise ValueError("policy head produced non-finite mean/std (torch Normal would have rejected them)")
        return m

    # ------------------------------------------------------------------ loops
    def run_training_loop(self, num_episodes: int, logger=None, tqdm_disable: bool = False, print_rewards: bool = False) -> Dict[str, float]:
        """reference: agent.py:329-418."""
        active_logger = logger or self.logger
        tr, lg = self.config["train"], self.config["logger"]
        update_every = tr.get("update_frequency", 1)
        grad_steps = tr.get("gradient_steps_per_update", 1)
        window = deque(maxlen=100)
        best_avg, avg_return = -float("inf"), 0.0
        total_episodes = total_steps = 0
        for episode in tqdm(range(num_episodes), disable=tqdm_disable):
            state, _ = self.env.reset()
            done, ep_return, ep_steps = False, 0.0, 0
            total_episodes += 1
            while not done:
                action = self.select_action(state)
                next_state, reward, terminated, truncated, _ = self.env.step(action)
                done = terminated or truncated
                self.store_transition(state, action, reward, next_state, done)
                state = next_state
                ep_return += reward
                ep_steps += 1
                total_steps += 1
                if self.can_update() and total_steps % update_every == 0:
                    self.training_steps(grad_steps) if grad_steps > 1 else self.training_step()
                if active_logger is not None and lg["log_q_values"]:
                    self._log_q_values(np.asarray(state, np.float32)[None], np.asarray(action, np.float32)[None], active_logger, total_steps)
            window.append(ep_return)
            avg_return = float(np.mean(window))
            best_avg = max(best_avg, avg_return)
            if active_logger is not None and lg["log_episode_stats"]:
                active_logger.log_episode_metrics(episode_idx=episode, reward=ep_return, length=ep_steps)
            if print_rewards:
                print(f"Episode {episode}, Return: {ep_return:.2f}, Average Return(last 100 episodes): {avg_return:.2f}")
        metrics = {"total_episodes": total_episodes, "best_avg_return": best_avg, "final_avg_return": avg_return}
        if active_logger is not None:
            active_logger.log_hparams(self.config, metrics)
        if lg["save_model"]["enabled"]:
            save_path = lg["save_model"]["path"]
            if save_path is None:
                save_path = active_logger.run_dir
            else:
                os.makedirs(save_path, exist_ok=True)
            model_path = os.path.join(save_path, "sac_agent.pth")
            self.save_agent(model_path)
            print(f"Agent saved to {model_path}")
        if active_logger is not None and lg["log_episode_stats"]:
            from .utils.logger_utils import save_lengths, save_rewards
            save_rewards(active_logger.run_dir, active_logger.episode_rewards)
            save_lengths(active_logger.run_dir, active_logger.episode_lengths)
        return metrics

    def eval_agent(self, num_episodes: int, render_mode: Optional[str] = None, tqdm_disable: bool = False,
                   print_returns: bool = False, writer=None) -> float:
        """reference: agent.py:420-460 -- deterministic rollouts."""
        eval_env = self._get_render_environment(render_mode)
        total = 0.0
        for episode in tqdm(range(num_episodes), disable=tqdm_disable):
            state, _ = eval_env.reset()
            done, ep_return, length = False, 0.0, 0
            while not done:
                state, reward, terminated, truncated, _ = eval_env.step(self.select_action(state, deterministic=True))
                done = terminated or truncated
                ep_return += reward
                length += 1
            total += ep_return
            if print_returns:
                print(f"Evaluation Episode {episode}, Return: {ep_return:.2f}")
            if writer is not None:
                writer.add_scalar("Eval/Episode/Return", ep_return, episode)
                writer.add_scalar("Eval/Episode/Length", length, episode)
        avg = total / num_episodes
        if print_returns:
            print(f"Average Return over {num_episodes} episodes: {avg:.2f}")
        if eval_env is not self.env:
            eval_env.close()
        return avg

    def _get_render_environment(self, render_mode: Optional[str]):
        """reference: agent.py:462-491."""
        if render_mode is None or getattr(self.env, "render_mode", None) == render_mode:
            return self.env
        spec = getattr(self.env, "spec", None)
        if not (spec and getattr(spec, "id", None)):
            print("Warning: Cannot create new env for rendering as env.spec.id is not available. Using original env.")
            return self.env
        try:
            import gymnasium as gym
            print(f"Creating new environment for evaluation with render_mode='{render_mode}'")
            eval_env = gym.make(spec.id, render_mode=render_mode)
            seed = self.config["train"].get("seed")
            if seed is not None:
                eval_env.reset(seed=seed)
                eval_env.action_space.seed(seed)
            return eval_env
        except Exception as e:  # noqa: BLE001
            print(f"Warning: Failed to create new env for rendering: {e}. Using original env.")
            return self.env

    def _log_q_values(self, states: Any, actions: Any, logger, step: int) -> None:
        """reference: agent.py:493-500."""
        q1, q2 = self.engine.q_values_host(np.asarray(states, np.float32), np.asarray(actions, np.float32))
        logger.log_q_values(float(q1.mean()), float(q2.mean()), step)

    def _infer_env_name(self, env) -> str:
        spec = getattr(env, "spec", None)
        if spec is not None and getattr(spec, "id", None):
            return spec.id
        return env.__class__.__name__

    def show_config(self, indent: int = 4) -> None:
        pprint.PrettyPrinter(indent=indent).pprint(self.config)

    def print_net_architectures(self) -> None:
        print("Policy Network Architecture:")
        print(self.policy_net)
        print("\nQ-Network 1 Architecture:")
        print(self.q_net1)
        print("\nQ-Network 2 Architecture:")
        print(self.q_net2)

    # ------------------------------------------------------------------ checkpoint (schema of agent.py:521-554)
    def save_agent(self, filepath: str) -> None:
        self.engine.sync()
        snap = lambda sd: {k: v.detach().clone() for k, v in sd.items()}

        def snap_opt(opt):
            sd = opt.state_dict()
            sd["state"] = {i: {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in st.items()} for i, st in sd["state"].items()}
            return sd

        ck = {
            "policy_net_state_dict": snap(self.policy_net.state_dict()),
            "q_net1_state_dict": snap(self.q_net1.state_dict()),
            "q_net2_state_dict": snap(self.q_net2.state_dict()),
            "q_net1_target_state_dict": snap(self.q_net1_target.state_dict()),
            "q_net2_target_state_dict": snap(self.q_net2_target.state_dict()),
            "policy_optimizer_state_dict": snap_opt(self.policy_optimizer),
            "q1_optimizer_state_dict": snap_opt(self.q1_optimizer),
            "q2_optimizer_state_dict": snap_opt(self.q2_optimizer),
        }
        if self.auto_entropy:
            ck["log_alpha"] = self.log_alpha.detach().clone()
            ck["alpha_optimizer_state_dict"] = snap_opt(self.alpha_optimizer)
        torch.save(ck, filepath)

    # ------------------------------------------------------------------ exact resume (SURVEY 8f-3; the reference cannot)
    def save_snapshot(self, filepath: str) -> None:
        """Everything a bit-exact continuation needs: the engine's scalar / parameter / optimiser / target blocks as one
        arena slice, the replay ring image, the rollout-noise counter and the host generators the host-RNG path consumes
        (Python ``random``, torch CPU, numpy). ``save_agent`` stays the reference-compatible checkpoint."""
        import random
        self.engine.sync()
        eng = self.engine
        end = eng.layout["block.targets"][0] + eng.layout["block.targets"][2]       # scalars | params | m | v | g | targets
        snap = {
            "format": "sacx-snapshot-1",
            "arena_head": eng.arena[:end].detach().cpu(),
            "act_counter": int(eng.lib.sacx_agent_act_counter(eng.h, -1)),
            "seed": int(self.config["train"]["seed"]),          # keys the device index / normal streams
            "ring": self.replay_buffer.image() if self.replay_buffer.handle is not None else None,
            "ring_dims": (self.replay_buffer.capacity, self.replay_buffer.obs_dim, self.replay_buffer.act_dim),
            "python_random": random.getstate(),
            "torch_rng": torch.get_rng_state(),
            "numpy_rng": np.random.get_state(),
        }
        if self.per is not None:                   # prioritized replay: priorities by ring slot and p_max
            leaves, p_max = self.replay_buffer.slot_priorities()
            snap["per"] = {"leaves": leaves.cpu(), "p_max": p_max}
        torch.save(snap, filepath)

    def load_snapshot(self, filepath: str) -> None:
        import random
        snap = torch.load(filepath, map_location="cpu", weights_only=False)
        if snap.get("format") != "sacx-snapshot-1":
            raise ValueError("not a sacx snapshot")
        if int(snap["seed"]) != int(self.config["train"]["seed"]):
            raise ValueError("snapshot was taken with train.seed=%d: build the agent from the same config to resume" % snap["seed"])
        if self.per is not None and snap.get("per") is None:
            raise ValueError("snapshot has no replay priorities: it was taken without buffer.prioritized")
        eng = self.engine
        eng.sync()
        head = snap["arena_head"]
        end = eng.layout["block.targets"][0] + eng.layout["block.targets"][2]
        if head.numel() != end:
            raise ValueError("snapshot was taken with different network shapes")
        eng.arena[:end].copy_(head.to(eng.arena.device))
        eng.lib.sacx_agent_act_counter(eng.h, int(snap["act_counter"]))
        if snap["ring"] is not None:
            cap, od, ad = snap["ring_dims"]
            if self.replay_buffer.handle is None:
                self.replay_buffer._allocate(int(od), int(ad))
                self.engine.attach_ring(self.replay_buffer)
            self.replay_buffer.load_image(snap["ring"])
        if self.per is not None:
            self.replay_buffer.load_slot_priorities(snap["per"]["leaves"], snap["per"]["p_max"])
        random.setstate(snap["python_random"])
        torch.set_rng_state(snap["torch_rng"])
        np.random.set_state(snap["numpy_rng"])
        eng.sync()

    def load_agent(self, filepath: str, reference_temperature_semantics: bool = False) -> None:
        """reference: agent.py:538-554. Accepts the reference's own files, including the (1,) float32 ``log_alpha`` of the
        shipped checkpoints (today's reference writes a 0-dim float64).

        One deliberate difference, off by default: in the reference ``load_agent`` REBINDS ``self.log_alpha`` to the loaded
        tensor while ``alpha_optimizer`` keeps the tensor made in ``__init__`` as its parameter, so after a load the
        temperature never moves again (alpha stays exp(loaded log_alpha)). Here the loaded value and optimiser state go into
        the live tensor and tuning continues. ``reference_temperature_semantics=True`` reproduces the reference (temperature
        frozen after the load) -- used by the parity tests that continue a reference run from a checkpoint."""
        ck = torch.load(filepath, map_location=self.device)
        self.engine.sync()
        self.policy_net.load_state_dict(ck["policy_net_state_dict"])
        self.q_net1.load_state_dict(ck["q_net1_state_dict"])
        self.q_net2.load_state_dict(ck["q_net2_state_dict"])
        self.q_net1_target.load_state_dict(ck["q_net1_target_state_dict"])
        self.q_net2_target.load_state_dict(ck["q_net2_target_state_dict"])
        self.policy_optimizer.load_state_dict(ck["policy_optimizer_state_dict"])
        self.q1_optimizer.load_state_dict(ck["q1_optimizer_state_dict"])
        self.q2_optimizer.load_state_dict(ck["q2_optimizer_state_dict"])
        if self.auto_entropy:
            la = torch.as_tensor(ck["log_alpha"]).detach()
            with torch.no_grad():
                self.log_alpha.copy_(la.to(self.device).double().reshape(-1)[0])
            self.alpha_optimizer.load_state_dict(ck["alpha_optimizer_state_dict"])
            lr = abs(float(self.engine.view("scal.alpha_lr").item())) or float(self.config["sac"]["alpha_lr"])
            self.engine.view("scal.alpha_lr").fill_(-lr if reference_temperature_semantics else lr)
        torch.cuda.synchronize(self.device)
        self.engine.refresh_alpha()
        if self.auto_entropy and la.dtype == torch.float32:
            # the reference's alpha = exp(log_alpha) is evaluated in the loaded tensor's dtype
            a32 = float(torch.exp(la.reshape(-1)[0].float()))
            self.engine.view("scal.alpha").fill_(a32)
            self.engine.view("scal.alpha_f32").fill_(a32)
