"""Device-resident replay ring behind the reference's ReplayBuffer API.

Reference: /root/reference/sac/replay_buffer.py -- ``Transition`` (:6-8), ``ReplayBuffer.__init__``
(:12-19, ``deque(maxlen=capacity)``), ``push`` (:21-30), ``sample`` (:32-39, ``random.sample`` on the
deque, ``ValueError`` when under-filled), ``__len__`` (:41-42).

Here the storage is a ring of packed records ``[s | s2 | a | r | d]`` in HBM owned by libsacx (``sacx_ring_*``): pushes go
through a pinned host staging block, sampling is a coalesced gather kernel.  The sampling *semantics*
are the reference's: ``sample`` draws ``random.sample(range(len), batch_size)`` from Python's global
Mersenne Twister -- the very index stream ``random.sample(deque, k)`` consumes (SURVEY F3) -- and maps
logical deque positions (0 = oldest survivor) to ring slots on the device.
"""
from __future__ import annotations

import ctypes as C
import math
import random
from collections import namedtuple
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _engine as E

Transition = namedtuple("Transition", ("state", "action", "reward", "next_state", "done"))


class _Occupancy:
    """Stand-in for the reference's ``.memory`` deque: callers only ever take ``len()`` of it."""

    def __init__(self, owner: "ReplayBuffer"):
        self._owner = owner

    def __len__(self) -> int:
        return len(self._owner)


def sample_range(n: int, k: int):
    """``random.sample(range(n), k)`` of CPython 3.12, bit for bit, in a few bulk draws instead of k Python-level loops.

    The stdlib's set-based branch (n larger than its small-population threshold) is a filter over the Mersenne Twister's
    32-bit outputs: ``_randbelow(n)`` keeps the top ``n.bit_length()`` bits of a word and rejects values >= n, and a
    value already selected is rejected too. ``getrandbits(32 * w)`` returns the same w words (least significant first),
    so drawing exactly as many words as selections are still missing never consumes a word the stdlib loop would not
    have consumed: the global generator ends in the same state. Other cases fall back to ``random.sample``."""
    bits = int(n).bit_length()
    setsize = 21
    if k > 5:
        setsize += 4 ** math.ceil(math.log(k * 3, 4))
    if not (0 < k <= n) or n <= setsize or bits > 32 or type(random.getrandbits.__self__) is not random.Random:
        return random.sample(range(n), k)
    getrandbits = random.getrandbits
    # Rounds of bulk draws. The stdlib loop consumes one 32-bit word per attempt and keeps attempting until k positions are
    # selected, so drawing exactly as many words as selections are still missing never reads a word it would not have read;
    # the accept/reject rule itself (value >= n, value selected before) runs in libsacx (sacx_index_filter, plain host code).
    lib = E.load()
    out = np.empty(k, dtype=np.int64)
    have = 0
    while have < k:
        need = k - have
        have = lib.sacx_index_filter(getrandbits(32 * need).to_bytes(4 * need, "little"), need, n, bits, out.ctypes.data, have, k)
        if have < 0:
            raise RuntimeError("sacx_index_filter rejected its arguments")
    return out                                                # int64 array (what the gather takes); same values as the stdlib's list


class ReplayBuffer:
    def __init__(self, capacity: int, obs_dim: Optional[int] = None, act_dim: Optional[int] = None,
                 device: Optional[str] = None, n_agents: int = 1):
        """capacity: maximum number of stored transitions (oldest evicted first).

        ``obs_dim`` / ``act_dim`` are optional: the reference constructor does not know them
        (replay_buffer.py:12, agent.py:29), so the ring is allocated lazily on the first push.
        """
        self.capacity = int(capacity)
        self.memory = _Occupancy(self)
        self.n_agents = int(n_agents)
        self.device = torch.device(device) if device is not None else None
        self.obs_dim = self.act_dim = None
        self._h = None
        self._store = None
        if obs_dim is not None and act_dim is not None:
            self._allocate(int(obs_dim), int(act_dim))

    # ------------------------------------------------------------------ native handle
    def _allocate(self, obs_dim: int, act_dim: int) -> None:
        E.require_cuda()
        lib = E.load()
        if self.device is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("the replay ring is device-resident: ReplayBuffer needs a CUDA device")
        self.obs_dim, self.act_dim = obs_dim, act_dim
        nbytes = lib.sacx_ring_bytes(obs_dim, act_dim, self.capacity, self.n_agents)
        with torch.cuda.device(self.device):
            self._store = torch.empty(nbytes // 4, dtype=torch.float32, device=self.device)
            h = C.c_void_p()
            E.check(lib.sacx_ring_create(obs_dim, act_dim, self.capacity, self.n_agents, self._store.data_ptr(), C.byref(h)))
        self._h = h
        self._lib = lib

    @property
    def handle(self):
        return self._h

    def __del__(self):
        try:
            if self._h is not None:
                self._lib.sacx_ring_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ reference API
    def push(self, state, action, reward, next_state, done, agent: int = 0) -> None:
        """Store one transition (reference: replay_buffer.py:21-30). Values are cast to float32,
        exactly the cast the reference applies at sample time (agent.py:171-185)."""
        s = np.ascontiguousarray(state, dtype=np.float32).reshape(-1)
        a = np.ascontiguousarray(action, dtype=np.float32).reshape(-1)
        s2 = np.ascontiguousarray(next_state, dtype=np.float32).reshape(-1)
        if self._h is None:
            self._allocate(s.size, a.size)
        if s.size != self.obs_dim or s2.size != self.obs_dim or a.size != self.act_dim:
            raise ValueError("transition shape does not match the buffer's (obs_dim, act_dim)")
        E.check(self._lib.sacx_ring_push_host(self._h, agent, s.ctypes.data, a.ctypes.data, float(reward),
                                              s2.ctypes.data, 1.0 if done else 0.0))

    add = push          # BASELINE.json calls it "add"; the reference method is ``push``

    def push_batch(self, states, actions, rewards, next_states, dones, agent: int = 0) -> None:
        """n transitions from host arrays in one call."""
        s = np.ascontiguousarray(states, dtype=np.float32)
        a = np.ascontiguousarray(actions, dtype=np.float32)
        s2 = np.ascontiguousarray(next_states, dtype=np.float32)
        r = np.ascontiguousarray(rewards, dtype=np.float32).reshape(-1)
        d = np.ascontiguousarray(dones, dtype=np.float32).reshape(-1)
        n = r.shape[0]
        if self._h is None:
            self._allocate(s.reshape(n, -1).shape[1], a.reshape(n, -1).shape[1])
        self._check_rows(n, s.size, a.size, s2.size, d.shape[0])
        E.check(self._lib.sacx_ring_push_n_host(self._h, agent, n, s.ctypes.data, a.ctypes.data, r.ctypes.data,
                                                s2.ctypes.data, d.ctypes.data))

    def push_device(self, states: torch.Tensor, actions: torch.Tensor, rewards: torch.Tensor,
                    next_states: torch.Tensor, dones: torch.Tensor, agent: int = 0) -> None:
        """n transitions that already live on the device (no host bounce)."""
        f = lambda t: t.to(device=self.device, dtype=torch.float32).contiguous()
        s, a, r, s2, d = f(states), f(actions), f(rewards).reshape(-1), f(next_states), f(dones).reshape(-1)
        n = r.shape[0]
        if self._h is None:
            self._allocate(s.reshape(n, -1).shape[1], a.reshape(n, -1).shape[1])
        self._check_rows(n, s.numel(), a.numel(), s2.numel(), d.shape[0])
        E.check(self._lib.sacx_ring_push_n_dev(self._h, agent, n, s.data_ptr(), a.data_ptr(), r.data_ptr(),
                                               s2.data_ptr(), d.data_ptr()))

    def _check_rows(self, n: int, s_elems: int, a_elems: int, s2_elems: int, d_elems: int) -> None:
        """the native push reads n rows of (obs_dim | act_dim | 1 | obs_dim | 1) floats through raw pointers: refuse anything else"""
        if s_elems != n * self.obs_dim or s2_elems != n * self.obs_dim or a_elems != n * self.act_dim or d_elems != n:
            raise ValueError(f"push of {n} transitions: expected states/next_states [{n}, {self.obs_dim}], actions [{n}, {self.act_dim}], "
                             f"rewards/dones [{n}]")

    def __len__(self) -> int:
        return 0 if self._h is None else int(self._lib.sacx_ring_len(self._h, 0))

    def size(self, agent: int = 0) -> int:
        return 0 if self._h is None else int(self._lib.sacx_ring_len(self._h, agent))

    def _require(self, batch_size: int, agent: int = 0) -> None:
        n = self.size(agent)
        if n < batch_size:
            raise ValueError(
                f"Not enough samples in the replay buffer to sample {batch_size} transitions. Current size: {n}")

    def draw_indices(self, batch_size: int, agent: int = 0):
        """The reference's index stream: k distinct logical positions from the global ``random``
        (``random.sample(self.memory, k)``, replay_buffer.py:39) -- same values, same generator state afterwards."""
        self._require(batch_size, agent)
        return sample_range(self.size(agent), batch_size)

    def sample(self, batch_size: int) -> List[Transition]:
        """Legacy list-of-Transition result (reference: replay_buffer.py:32-39)."""
        idx = np.asarray(self.draw_indices(batch_size), dtype=np.int64)
        s, a, r, s2, d = self.gather_host(idx)
        return [Transition(s[i], a[i], float(r[i]), s2[i], bool(d[i] != 0.0)) for i in range(batch_size)]

    # ------------------------------------------------------------------ exact-resume image
    def image(self) -> torch.Tensor:
        """The whole ring (headers with the push counters + packed records) as one CPU tensor."""
        E.check(self._lib.sacx_ring_flush(self._h))
        torch.cuda.synchronize(self.device)
        return self._store.detach().cpu()

    def load_image(self, img: torch.Tensor) -> None:
        if self._h is None or img.numel() != self._store.numel():
            raise ValueError("ring image does not match this buffer (capacity / obs_dim / act_dim / n_agents)")
        E.check(self._lib.sacx_ring_flush(self._h))
        self._store.copy_(img.to(self.device))
        torch.cuda.synchronize(self.device)
        E.check(self._lib.sacx_ring_resync(self._h))

    # ------------------------------------------------------------------ fast paths
    def gather_host(self, logical_idx: Sequence[int], agent: int = 0):
        idx = np.ascontiguousarray(logical_idx, dtype=np.int64)
        B = idx.shape[0]
        self._require(B, agent)
        s = np.empty((B, self.obs_dim), np.float32)
        a = np.empty((B, self.act_dim), np.float32)
        r = np.empty(B, np.float32)
        s2 = np.empty((B, self.obs_dim), np.float32)
        d = np.empty(B, np.float32)
        E.check(self._lib.sacx_ring_gather_host(self._h, agent, idx.ctypes.data, B, s.ctypes.data, a.ctypes.data,
                                                r.ctypes.data, s2.ctypes.data, d.ctypes.data))
        return s, a, r, s2, d

    def sample_tensors(self, batch_size: int, indices=None, agent: int = 0) -> Transition:
        """Batch as device tensors. ``indices``: logical positions (host sequence or device int64
        tensor); None draws them from the global ``random`` like the reference."""
        self._require(batch_size, agent)
        if indices is None:
            indices = self.draw_indices(batch_size, agent)
        if not torch.is_tensor(indices):
            host = np.asarray(indices, dtype=np.int64).reshape(-1)
            if host.size and (host.min() < 0 or host.max() >= self.size(agent)):      # logical positions of the deque: [0, len)
                raise ValueError("logical index out of range")
            indices = torch.as_tensor(host)
        # (a device tensor is not read back for validation -- that would put a sync into every gather; the kernels themselves
        #  never read outside the ring: a position outside [0, len) yields a zero row)
        idx = indices.to(device=self.device, dtype=torch.int64).contiguous().reshape(-1)
        B = idx.shape[0]
        if B != batch_size:
            raise ValueError(f"{B} indices given for a batch of {batch_size}")
        kw = dict(dtype=torch.float32, device=self.device)
        s, a = torch.empty(B, self.obs_dim, **kw), torch.empty(B, self.act_dim, **kw)
        r, s2, d = torch.empty(B, **kw), torch.empty(B, self.obs_dim, **kw), torch.empty(B, **kw)
        E.check(self._lib.sacx_ring_gather(self._h, agent, idx.data_ptr(), B, s.data_ptr(), a.data_ptr(), r.data_ptr(),
                                           s2.data_ptr(), d.data_ptr()))
        return Transition(s, a, r, s2, d)

    def device_indices(self, batch_size: int, seed: int, counter: int, agent: int = 0) -> torch.Tensor:
        """B distinct logical positions generated on the device (throughput mode's sampler)."""
        self._require(batch_size, agent)
        out = torch.empty(batch_size, dtype=torch.int64, device=self.device)
        E.check(self._lib.sacx_ring_sample_indices(self._h, agent, seed, counter, batch_size, out.data_ptr()))
        return out

    def flush(self) -> None:
        if self._h is not None:
            E.check(self._lib.sacx_ring_flush(self._h))


class PrioritizedReplayBuffer(ReplayBuffer):
    """Prioritized experience replay (Schaul et al., 2016) on the device ring: a sum/min tree over the ring's slots
    (``sacx_per_*``), proportional stratified sampling, importance weights ``w = (p / p_min)^-beta`` and priorities
    ``p = (|td| + eps)^alpha``. New transitions enter with the largest priority assigned so far (initially 1).

    ``sample_tensors(B, beta=None)`` returns ``(Transition, weights, indices)``: device tensors, ``indices`` are logical
    positions (0 = oldest) to hand back to ``update_priorities(indices, td_abs)``. Draws are keyed by ``seed`` and a call
    counter. Attached to a SAC agent (``buffer.prioritized``), the agent's own updates sample and refresh the tree on the
    device. ``sample`` and ``draw_indices`` stay the uniform stream of ``ReplayBuffer``."""

    def __init__(self, capacity: int, obs_dim: Optional[int] = None, act_dim: Optional[int] = None,
                 device: Optional[str] = None, alpha: float = 0.6, beta: float = 0.4, beta_steps: int = 0, eps: float = 1e-6,
                 max_batch: int = 65536, seed: int = 0):
        cfg = E.per_config({"buffer": {"prioritized": {"alpha": alpha, "beta": beta, "beta_steps": beta_steps, "eps": eps}}})
        self.alpha, self.beta, self.beta_steps, self.eps = cfg["alpha"], cfg["beta"], cfg["beta_steps"], cfg["eps"]
        self.max_batch, self.seed, self._draws = int(max_batch), int(seed), 0
        self._per = None
        super().__init__(capacity, obs_dim, act_dim, device=device)

    def _allocate(self, obs_dim: int, act_dim: int) -> None:
        super()._allocate(obs_dim, act_dim)
        h = C.c_void_p()
        E.check(self._lib.sacx_per_create(self._h, self.alpha, self.beta, self.beta_steps, self.eps, self.max_batch, C.byref(h)))
        self._per = h

    @property
    def per_handle(self):
        return self._per

    def __del__(self):
        try:
            if self._per is not None:
                self._lib.sacx_per_destroy(self._per)
                self._per = None
        except Exception:
            pass
        super().__del__()

    def sample_tensors(self, batch_size: int, beta: Optional[float] = None):
        self._require(batch_size)
        beta = self.beta if beta is None else float(beta)
        kw = dict(device=self.device)
        idx = torch.empty(batch_size, dtype=torch.int64, **kw)
        w = torch.empty(batch_size, dtype=torch.float32, **kw)
        E.check(self._lib.sacx_per_sample(self._per, int(batch_size), beta, None, self.seed, self._draws, idx.data_ptr(), w.data_ptr()))
        self._draws += 1
        return ReplayBuffer.sample_tensors(self, batch_size, idx), w, idx

    def sample_with_uniforms(self, u: torch.Tensor, beta: Optional[float] = None):
        """Indices and weights for given stratum offsets ``u`` in [0, 1) (row k draws (k + u_k) / B of the total priority)."""
        u = u.to(device=self.device, dtype=torch.float32).contiguous().reshape(-1)
        B = u.shape[0]
        beta = self.beta if beta is None else float(beta)
        idx = torch.empty(B, dtype=torch.int64, device=self.device)
        w = torch.empty(B, dtype=torch.float32, device=self.device)
        E.check(self._lib.sacx_per_sample(self._per, B, beta, u.data_ptr(), 0, 0, idx.data_ptr(), w.data_ptr()))
        return idx, w

    def update_priorities(self, indices, td_abs) -> None:
        idx = torch.as_tensor(indices).to(device=self.device, dtype=torch.int64).contiguous().reshape(-1)
        td = torch.as_tensor(td_abs).to(device=self.device, dtype=torch.float32).contiguous().reshape(-1)
        if idx.shape != td.shape:
            raise ValueError("indices and td_abs differ in length")
        if idx.numel():
            E.check(self._lib.sacx_per_update_priorities(self._per, idx.data_ptr(), td.data_ptr(), idx.numel()))

    def slot_priorities(self):
        """(priorities by ring slot [capacity], 0 = empty slot; p_max), pending writes applied."""
        leaves = torch.empty(self.capacity, dtype=torch.float32, device=self.device)
        pm = C.c_float()
        E.check(self._lib.sacx_per_priorities(self._per, leaves.data_ptr(), C.byref(pm)))
        return leaves, float(pm.value)

    def priorities(self) -> torch.Tensor:
        """Priority of every stored transition in logical order (0 = oldest), a device tensor of length len(self)."""
        leaves, _ = self.slot_priorities()
        n, pushes = len(self), int(self._lib.sacx_ring_pushes(self._h, 0))
        oldest = (pushes - self.capacity) % self.capacity if pushes > self.capacity else 0
        return leaves[(oldest + torch.arange(n, device=self.device)) % self.capacity]

    def load_slot_priorities(self, leaves: torch.Tensor, p_max: float) -> None:
        leaves = leaves.to(device=self.device, dtype=torch.float32).contiguous()
        if leaves.numel() != self.capacity:
            raise ValueError("priority image does not match this buffer's capacity")
        E.check(self._lib.sacx_per_load_priorities(self._per, leaves.data_ptr(), float(p_max)))
