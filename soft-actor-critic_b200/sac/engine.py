"""``UpdateEngine``: Python handle on one libsacx agent (or a population of agents).

Owns the packed device arena (a torch float32 tensor, so every named tensor of the engine is a
zero-copy torch view: parameters, targets, Adam moments, gradients, temperature scalars, batch and
activation scratch) and forwards the update calls of include/sacx.h.  torch is plumbing here --
device memory, streams, views -- the arithmetic is in the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _engine as E


class UpdateEngine:
    def __init__(self, obs_dim: int, act_dim: int, config: dict, device="cuda", n_agents: int = 1,
                 ctas_per_agent: int = 0, dp_world: int = 1, dp_rank: int = 0, batch_size: Optional[int] = None,
                 agent_id_base: int = 0):
        E.require_cuda()
        self.lib = E.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"train.device={device!r}: the SAC update engine is CUDA-only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.obs_dim, self.act_dim, self.n_agents = int(obs_dim), int(act_dim), int(n_agents)
        self.cfg = E.make_config(obs_dim, act_dim, config, n_agents, ctas_per_agent, dp_world, dp_rank, batch_size, agent_id_base)
        self.batch_size = int(self.cfg.batch_size)
        floats = C.c_int64()
        E.check(self.lib.sacx_agent_arena_floats(C.byref(self.cfg), C.byref(floats)))
        self.stride = int(floats.value)
        with torch.cuda.device(self.device):
            self.arena = torch.zeros(self.stride * self.n_agents, dtype=torch.float32, device=self.device)
            h = C.c_void_p()
            E.check(self.lib.sacx_agent_create(C.byref(self.cfg), self.arena.data_ptr(), C.byref(h)))
        self.h = h
        n = C.c_int32()
        E.check(self.lib.sacx_agent_layout(self.h, None, 0, C.byref(n)))
        descs = (E.SacxTensorDesc * n.value)()
        E.check(self.lib.sacx_agent_layout(self.h, descs, n.value, C.byref(n)))
        self.layout: Dict[str, Tuple[int, int, int, int, int]] = {
            d.name.decode(): (int(d.offset), int(d.rows), int(d.cols), int(d.ld), int(d.dtype)) for d in descs}
        self.ring = None
        self.per = None
        self._stream = None
        self._metrics = E.SacxMetrics()

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None:
                self.lib.sacx_agent_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ views
    def view(self, name: str, agent: int = 0) -> torch.Tensor:
        off, rows, cols, ld, dtype = self.layout[name]
        base = agent * self.stride + off
        if dtype == 0:
            flat = self.arena[base: base + rows * ld]
            t = flat.view(rows, ld)[:, :cols] if ld != cols else flat.view(rows, cols)
            return t
        words = self.arena[base: base + 2 * rows * ld]
        t = words.view(torch.float64 if dtype == 1 else torch.int64)
        return t.view(rows, ld)[:, :cols] if rows > 1 else t[:cols]

    def views(self, agent: int = 0) -> Dict[str, torch.Tensor]:
        return {k: self.view(k, agent) for k in self.layout}

    def population_view(self, name: str) -> torch.Tensor:
        """[n_agents, rows, cols] strided view of one named f32 tensor across the population."""
        off, rows, cols, ld, dtype = self.layout[name]
        assert dtype == 0
        return torch.as_strided(self.arena, (self.n_agents, rows, cols), (self.stride, ld, 1), off)

    # ------------------------------------------------------------------ plumbing
    def _sync_stream(self) -> None:
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self._stream:
            E.check(self.lib.sacx_agent_set_stream(self.h, s))
            if self.ring is not None and self.ring.handle is not None:
                E.check(self.lib.sacx_ring_set_stream(self.ring.handle, s))
            self._stream = s

    def attach_ring(self, ring) -> None:
        self.ring = ring
        E.check(self.lib.sacx_agent_attach_ring(self.h, ring.handle if ring is not None else None))
        self._stream = None

    def attach_per(self, buf) -> None:
        """Prioritized replay: ``buf`` a PrioritizedReplayBuffer (the attached ring's), or None for uniform sampling."""
        E.check(self.lib.sacx_agent_attach_per(self.h, buf.per_handle if buf is not None else None))
        self.per = buf

    def reset_state(self) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_agent_reset_state(self.h))

    def refresh_alpha(self) -> None:
        E.check(self.lib.sacx_agent_refresh_alpha(self.h))

    def grid(self) -> Tuple[int, int, int]:
        a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
        E.check(self.lib.sacx_agent_grid(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def path(self) -> Tuple[str, str]:
        """("rowpar" | "tiles", reason): which kernel runs ``update`` (include/sacx.h: sacx_agent_path)."""
        buf = C.create_string_buffer(128)
        rc = self.lib.sacx_agent_path(self.h, buf, 128)
        if rc < 0:
            E.check(rc)
        return ("rowpar" if rc == 1 else "tiles"), buf.value.decode()

    def tensor_core(self) -> Tuple[bool, str, int]:
        """(enabled, reason when not, tensor-core kernel launches so far) -- include/sacx.h: sacx_agent_tc."""
        buf = C.create_string_buffer(128)
        n = C.c_int64(0)
        rc = self.lib.sacx_agent_tc(self.h, buf, 128, C.byref(n))
        if rc < 0:
            E.check(rc)
        return rc == 1, buf.value.decode(), int(n.value)

    def sync(self) -> None:
        E.check(self.lib.sacx_sync(self.h))

    def launch_count(self) -> int:
        return int(self.lib.sacx_launch_count(self.h))

    # ------------------------------------------------------------------ updates
    def update(self, idx: Optional[torch.Tensor] = None, eps1: Optional[torch.Tensor] = None,
               eps2: Optional[torch.Tensor] = None, n_steps: int = 1, staged: bool = False) -> None:
        """n_steps fused updates; device tensors or None (device RNG)."""
        self._sync_stream()
        fn = self.lib.sacx_update_staged if staged else self.lib.sacx_update
        E.check(fn(self.h, E.ptr(idx), E.ptr(eps1), E.ptr(eps2), int(n_steps)))

    def update_host(self, idx: Optional[np.ndarray], eps1: Optional[np.ndarray], eps2: Optional[np.ndarray],
                    n_steps: int = 1, want_metrics: bool = True) -> Optional[dict]:
        """Same through host buffers: H2D copies, update, D2H of the metrics (the e2e path)."""
        self._sync_stream()
        m = C.byref(self._metrics) if want_metrics else None
        E.check(self.lib.sacx_update_host(self.h, E.ptr(idx), E.ptr(eps1), E.ptr(eps2), int(n_steps), m))
        return self._metrics.as_dict() if want_metrics else None

    def update_host_pipelined(self, idx, eps1, eps2, n_steps: int = 1) -> Optional[dict]:
        """Submit this update and return the metrics of the previous submission (None on the first call): the
        host draws the next index stream / normals while the GPU runs the current update."""
        self._sync_stream()
        have = C.c_int32(0)
        E.check(self.lib.sacx_update_host_pipelined(self.h, E.ptr(idx), E.ptr(eps1), E.ptr(eps2), int(n_steps),
                                                    C.byref(self._metrics), C.byref(have)))
        return self._metrics.as_dict() if have.value else None

    def update_host_flush(self) -> dict:
        E.check(self.lib.sacx_update_host_flush(self.h, C.byref(self._metrics)))
        return self._metrics.as_dict()

    def sample_batch(self, idx: Optional[torch.Tensor] = None) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_sample_batch(self.h, E.ptr(idx)))

    def load_batch(self, s=None, a=None, r=None, s2=None, d=None) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_load_batch(self.h, E.ptr(s), E.ptr(a), E.ptr(r), E.ptr(s2), E.ptr(d)))

    def target(self, eps1=None, y_out=None) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_target(self.h, E.ptr(eps1), E.ptr(y_out)))

    def critic_step(self, y=None, grads_only: bool = False) -> None:
        self._sync_stream()
        fn = self.lib.sacx_critic_grads if grads_only else self.lib.sacx_critic_step
        E.check(fn(self.h, E.ptr(y)))

    def actor_step(self, eps2=None, logpi_out=None, grads_only: bool = False) -> None:
        self._sync_stream()
        fn = self.lib.sacx_actor_grads if grads_only else self.lib.sacx_actor_step
        E.check(fn(self.h, E.ptr(eps2), E.ptr(logpi_out)))

    def alpha_step(self, logpi=None, want_metrics: bool = False) -> Optional[dict]:
        self._sync_stream()
        m = C.byref(self._metrics) if want_metrics else None
        E.check(self.lib.sacx_alpha_step(self.h, E.ptr(logpi), m))
        return self._metrics.as_dict() if want_metrics else None

    def polyak(self) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_polyak(self.h))

    def apply_grads(self, which: int, polyak: bool = False) -> None:
        self._sync_stream()
        E.check(self.lib.sacx_apply_grads(self.h, int(which), 1 if polyak else 0))

    def act(self, states: torch.Tensor, eps: Optional[torch.Tensor] = None, deterministic: bool = False, agent: int = 0) -> torch.Tensor:
        self._sync_stream()
        s = states.to(device=self.device, dtype=torch.float32).contiguous().view(-1, self.obs_dim)
        out = torch.empty(s.shape[0], self.act_dim, dtype=torch.float32, device=self.device)
        E.check(self.lib.sacx_act(self.h, agent, s.data_ptr(), s.shape[0], E.ptr(eps), 1 if deterministic else 0, out.data_ptr()))
        return out

    def act_population(self, states: torch.Tensor, eps: Optional[torch.Tensor] = None, deterministic: bool = False) -> torch.Tensor:
        """states [n_agents, n, obs] (device) -> actions [n_agents, n, act]: every agent's policy on its own states, one launch."""
        self._sync_stream()
        s = states.to(device=self.device, dtype=torch.float32).contiguous().view(self.n_agents, -1, self.obs_dim)
        n = s.shape[1]
        out = torch.empty(self.n_agents, n, self.act_dim, device=self.device, dtype=torch.float32)
        e = None if eps is None else eps.to(device=self.device, dtype=torch.float32).contiguous()
        E.check(self.lib.sacx_act_population(self.h, E.ptr(s), n, E.ptr(e), 1 if deterministic else 0, E.ptr(out)))
        return out

    def act_host(self, state: np.ndarray, eps: Optional[np.ndarray] = None, deterministic: bool = False, agent: int = 0) -> np.ndarray:
        self._sync_stream()
        s = np.ascontiguousarray(state, dtype=np.float32).reshape(-1, self.obs_dim)
        out = np.empty((s.shape[0], self.act_dim), np.float32)
        e = None if eps is None else np.ascontiguousarray(eps, dtype=np.float32)
        E.check(self.lib.sacx_act_host(self.h, agent, s.ctypes.data, s.shape[0], E.ptr(e), 1 if deterministic else 0, out.ctypes.data))
        return out

    def q_values(self, states: torch.Tensor, actions: torch.Tensor, agent: int = 0):
        self._sync_stream()
        s = states.to(device=self.device, dtype=torch.float32).contiguous().view(-1, self.obs_dim)
        a = actions.to(device=self.device, dtype=torch.float32).contiguous().view(-1, self.act_dim)
        q1 = torch.empty(s.shape[0], dtype=torch.float32, device=self.device)
        q2 = torch.empty_like(q1)
        E.check(self.lib.sacx_q_values(self.h, agent, s.data_ptr(), a.data_ptr(), s.shape[0], q1.data_ptr(), q2.data_ptr()))
        return q1, q2

    def q_values_host(self, state: np.ndarray, action: np.ndarray, agent: int = 0):
        self._sync_stream()
        s = np.ascontiguousarray(state, dtype=np.float32).reshape(-1, self.obs_dim)
        a = np.ascontiguousarray(action, dtype=np.float32).reshape(-1, self.act_dim)
        q1 = np.empty(s.shape[0], np.float32)
        q2 = np.empty(s.shape[0], np.float32)
        E.check(self.lib.sacx_q_values_host(self.h, agent, s.ctypes.data, a.ctypes.data, s.shape[0], q1.ctypes.data, q2.ctypes.data))
        return q1, q2

    # ------------------------------------------------------------------ population-based training (include/sacx.h: sacx_pbt_*)
    def pbt_state_floats(self) -> int:
        """float32 words of one packed learner state."""
        return int(self.lib.sacx_pbt_state_floats(self.h))

    @staticmethod
    def _ids(ids) -> np.ndarray:
        return np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1).astype(np.int32))

    @staticmethod
    def _records(records, n: int):
        if records is None:
            return None
        if len(records) != n:
            raise ValueError("one record per pair expected")
        return (E.SacxPbtRecord * n)(*records)

    def pbt_copy(self, src, dst, records=None) -> None:
        """Agent dst[i] takes the learner state of agent src[i] (local ids), then records[i]: one launch on the engine's stream."""
        self._sync_stream()
        s, d = self._ids(src), self._ids(dst)
        if len(s) != len(d):
            raise ValueError("pbt_copy: src and dst differ in length")
        E.check(self.lib.sacx_pbt_copy(self.h, s.ctypes.data, d.ctypes.data, len(d), self._records(records, len(d))))

    def pbt_pack(self, agents, buf: torch.Tensor) -> None:
        """buf[k] <- learner state of agent agents[k]; buf a contiguous float32 device tensor [len(agents), pbt_state_floats()]."""
        self._sync_stream()
        a = self._ids(agents)
        if buf.dtype != torch.float32 or not buf.is_contiguous() or buf.numel() < len(a) * self.pbt_state_floats():
            raise ValueError("pbt_pack: buffer must be a contiguous float32 tensor of len(agents) packed states")
        E.check(self.lib.sacx_pbt_pack(self.h, a.ctypes.data, len(a), E.ptr(buf)))

    def pbt_unpack(self, buf: torch.Tensor, slots, dst, records=None) -> None:
        """Agent dst[i] takes the packed state buf[slots[i]], then records[i]."""
        self._sync_stream()
        s, d = self._ids(slots), self._ids(dst)
        if len(s) != len(d):
            raise ValueError("pbt_unpack: slots and dst differ in length")
        if buf.dtype != torch.float32 or not buf.is_contiguous():
            raise ValueError("pbt_unpack: buffer must be a contiguous float32 tensor")
        n_slots = buf.numel() // max(self.pbt_state_floats(), 1)
        E.check(self.lib.sacx_pbt_unpack(self.h, E.ptr(buf), n_slots, s.ctypes.data, d.ctypes.data, len(d),
                                         self._records(records, len(d))))

    def metrics(self, agent: int = 0) -> dict:
        self._sync_stream()
        E.check(self.lib.sacx_get_metrics(self.h, agent, C.byref(self._metrics)))
        return self._metrics.as_dict()
