"""ctypes binding of libsacx.so (include/sacx.h) -- the only native dependency of this package.

There is deliberately no fallback: if the shared library is missing or no CUDA device is
present, importing is fine (so that host-side logic can be unit-tested) but the first call
that needs the engine raises ``RuntimeError``.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

SACX_MAX_HIDDEN = 8
SACX_MAX_ACT = 32

ACTIVATION_IDS = {"identity": 0, "relu": 1, "tanh": 2, "elu": 3, "leaky_relu": 4, "gelu": 5, "selu": 6}

SACX_OK = 0
SACX_ERR_INVALID = -1
SACX_ERR_UNDERFILLED = -2
SACX_ERR_CUDA = -3
SACX_ERR_ACTIVATION = -4
SACX_ERR_NONFINITE = -5
SACX_ERR_EMPTY_HIDDEN = -6


class SacxConfig(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32),
        ("n_hidden_pi", C.c_int32), ("hidden_pi", C.c_int32 * SACX_MAX_HIDDEN),
        ("n_hidden_q", C.c_int32), ("hidden_q", C.c_int32 * SACX_MAX_HIDDEN),
        ("act_hidden_pi", C.c_int32), ("act_out_pi", C.c_int32),
        ("act_hidden_q", C.c_int32), ("act_out_q", C.c_int32),
        ("batch_size", C.c_int32), ("auto_entropy_tuning", C.c_int32),
        ("n_agents", C.c_int32), ("ctas_per_agent", C.c_int32),
        ("log_std_min", C.c_float), ("log_std_max", C.c_float), ("action_scale", C.c_float),
        ("reserved_f", C.c_float),
        ("gamma", C.c_double), ("tau", C.c_double),
        ("alpha", C.c_double), ("actor_lr", C.c_double), ("critic_lr", C.c_double), ("alpha_lr", C.c_double),
        ("seed", C.c_uint64),
        ("dp_world", C.c_int32), ("dp_rank", C.c_int32),
        ("agent_id_base", C.c_int32), ("reserved_i", C.c_int32),
    ]


class SacxMetrics(C.Structure):
    _fields_ = [
        ("q1_loss", C.c_float), ("q2_loss", C.c_float), ("policy_loss", C.c_float), ("alpha_loss", C.c_float),
        ("alpha", C.c_float), ("log_alpha", C.c_float), ("q1_mean", C.c_float), ("q2_mean", C.c_float),
        ("logpi_mean", C.c_float), ("y_mean", C.c_float),
        ("nonfinite", C.c_int32), ("reserved", C.c_int32), ("updates", C.c_int64),
    ]

    def as_dict(self) -> Dict[str, float]:
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class SacxTensorDesc(C.Structure):
    _fields_ = [("name", C.c_char * 40), ("offset", C.c_int64), ("rows", C.c_int32), ("cols", C.c_int32),
                ("ld", C.c_int32), ("dtype", C.c_int32)]


# every symbol include/sacx.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I32, _I64, _U64, _F = C.c_int32, C.c_int64, C.c_uint64, C.c_float
SYMBOLS = {
    "sacx_last_error": (C.c_char_p, []),
    "sacx_version": (C.c_int, []),
    "sacx_device_count": (C.c_int, []),
    "sacx_sizeof_config": (C.c_int, []),
    "sacx_sizeof_metrics": (C.c_int, []),
    "sacx_sizeof_tensor_desc": (C.c_int, []),
    "sacx_activation_id": (C.c_int, [C.c_char_p]),
    "sacx_ring_bytes": (_I64, [_I32, _I32, _I64, _I32]),
    "sacx_ring_create": (C.c_int, [_I32, _I32, _I64, _I32, _P, C.POINTER(_P)]),
    "sacx_ring_destroy": (C.c_int, [_P]),
    "sacx_ring_set_stream": (C.c_int, [_P, _P]),
    "sacx_ring_push_host": (C.c_int, [_P, _I32, _P, _P, _F, _P, _F]),
    "sacx_ring_push_n_host": (C.c_int, [_P, _I32, _I64, _P, _P, _P, _P, _P]),
    "sacx_ring_push_n_dev": (C.c_int, [_P, _I32, _I64, _P, _P, _P, _P, _P]),
    "sacx_ring_flush": (C.c_int, [_P]),
    "sacx_ring_len": (_I64, [_P, _I32]),
    "sacx_ring_pushes": (_I64, [_P, _I32]),
    "sacx_ring_gather": (C.c_int, [_P, _I32, _P, _I32, _P, _P, _P, _P, _P]),
    "sacx_ring_gather_host": (C.c_int, [_P, _I32, _P, _I32, _P, _P, _P, _P, _P]),
    "sacx_ring_resync": (C.c_int, [_P]),
    "sacx_index_filter": (_I32, [C.c_char_p, _I32, _U64, _I32, _P, _I32, _I32]),
    "sacx_ring_sample_indices": (C.c_int, [_P, _I32, _U64, _U64, _I32, _P]),
    "sacx_per_create": (C.c_int, [_P, _F, _F, _I64, _F, _I32, C.POINTER(_P)]),
    "sacx_per_destroy": (C.c_int, [_P]),
    "sacx_per_sample": (C.c_int, [_P, _I32, _F, _P, _U64, _U64, _P, _P]),
    "sacx_per_update_priorities": (C.c_int, [_P, _P, _P, _I32]),
    "sacx_per_priorities": (C.c_int, [_P, _P, C.POINTER(_F)]),
    "sacx_per_load_priorities": (C.c_int, [_P, _P, _F]),
    "sacx_agent_attach_per": (C.c_int, [_P, _P]),
    "sacx_obs_create": (C.c_int, [_I32, _I32, _I32, _I32, C.POINTER(_P)]),
    "sacx_obs_destroy": (C.c_int, [_P]),
    "sacx_obs_dim": (_I32, [_P]),
    "sacx_obs_reset": (C.c_int, [_P, _P, _P, _P]),
    "sacx_obs_step": (C.c_int, [_P, _P, _P, _P, _F, _I32, _P, _I32, _P, _P]),
    "sacx_agent_arena_floats": (C.c_int, [C.POINTER(SacxConfig), C.POINTER(_I64)]),
    "sacx_agent_create": (C.c_int, [C.POINTER(SacxConfig), _P, C.POINTER(_P)]),
    "sacx_agent_destroy": (C.c_int, [_P]),
    "sacx_agent_set_stream": (C.c_int, [_P, _P]),
    "sacx_agent_attach_ring": (C.c_int, [_P, _P]),
    "sacx_agent_arena": (_P, [_P]),
    "sacx_agent_stride": (_I64, [_P]),
    "sacx_agent_layout": (C.c_int, [_P, C.POINTER(SacxTensorDesc), _I32, C.POINTER(_I32)]),
    "sacx_agent_reset_state": (C.c_int, [_P]),
    "sacx_agent_refresh_alpha": (C.c_int, [_P]),
    "sacx_agent_grid": (C.c_int, [_P, C.POINTER(_I32), C.POINTER(_I32), C.POINTER(_I32)]),
    "sacx_agent_path": (C.c_int, [_P, C.c_char_p, _I32]),
    "sacx_agent_act_counter": (_I64, [_P, _I64]),
    "sacx_agent_tc": (C.c_int, [_P, C.c_char_p, _I32, C.POINTER(_I64)]),
    "sacx_update": (C.c_int, [_P, _P, _P, _P, _I32]),
    "sacx_update_host": (C.c_int, [_P, _P, _P, _P, _I32, C.POINTER(SacxMetrics)]),
    "sacx_update_staged": (C.c_int, [_P, _P, _P, _P, _I32]),
    "sacx_update_host_pipelined": (C.c_int, [_P, _P, _P, _P, _I32, C.POINTER(SacxMetrics), C.POINTER(_I32)]),
    "sacx_update_host_flush": (C.c_int, [_P, C.POINTER(SacxMetrics)]),
    "sacx_sample_batch": (C.c_int, [_P, _P]),
    "sacx_load_batch": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "sacx_target": (C.c_int, [_P, _P, _P]),
    "sacx_critic_step": (C.c_int, [_P, _P]),
    "sacx_actor_step": (C.c_int, [_P, _P, _P]),
    "sacx_alpha_step": (C.c_int, [_P, _P, C.POINTER(SacxMetrics)]),
    "sacx_polyak": (C.c_int, [_P]),
    "sacx_critic_grads": (C.c_int, [_P, _P]),
    "sacx_actor_grads": (C.c_int, [_P, _P, _P]),
    "sacx_apply_grads": (C.c_int, [_P, _I32, _I32]),
    "sacx_act": (C.c_int, [_P, _I32, _P, _I32, _P, _I32, _P]),
    "sacx_act_population": (C.c_int, [_P, _P, _I32, _P, _I32, _P]),
    "sacx_act_host": (C.c_int, [_P, _I32, _P, _I32, _P, _I32, _P]),
    "sacx_q_values": (C.c_int, [_P, _I32, _P, _P, _I32, _P, _P]),
    "sacx_q_values_host": (C.c_int, [_P, _I32, _P, _P, _I32, _P, _P]),
    "sacx_get_metrics": (C.c_int, [_P, _I32, C.POINTER(SacxMetrics)]),
    "sacx_sync": (C.c_int, [_P]),
    "sacx_debug_profile": (C.c_int, [_P, _I32, _P, _I64, C.POINTER(_I32), C.POINTER(_I32)]),
    "sacx_launch_count": (_I64, [_P]),
}

_LIB: Optional[C.CDLL] = None


def lib_path() -> str:
    here = os.path.dirname(os.path.abspath(__file__))
    return os.environ.get("SACX_LIB", os.path.join(os.path.dirname(here), "lib", "libsacx.so"))


def load() -> C.CDLL:
    """Load libsacx.so and type every declared entry point. Raises RuntimeError when absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"libsacx.so not found at {path}: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "The SAC update engine is CUDA-only and has no Python/CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)           # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if (lib.sacx_sizeof_config() != C.sizeof(SacxConfig) or lib.sacx_sizeof_metrics() != C.sizeof(SacxMetrics)
            or lib.sacx_sizeof_tensor_desc() != C.sizeof(SacxTensorDesc)):
        raise RuntimeError("libsacx.so struct layout differs from the Python binding (stale build?)")
    _LIB = lib
    return lib


def check(rc: int) -> None:
    """Translate a status code into the exception class the reference raises in the same situation."""
    if rc == SACX_OK:
        return
    msg = load().sacx_last_error().decode("utf-8", "replace")
    if rc in (SACX_ERR_INVALID, SACX_ERR_UNDERFILLED, SACX_ERR_NONFINITE, SACX_ERR_EMPTY_HIDDEN):
        raise ValueError(msg)
    if rc == SACX_ERR_ACTIVATION:
        raise KeyError(msg)
    raise RuntimeError(f"libsacx: {msg} (status {rc})")


def require_cuda() -> None:
    lib = load()
    if lib.sacx_device_count() < 1:
        raise RuntimeError("no CUDA device visible: the B200 SAC engine has no CPU fallback for the update path")


def ptr(t) -> Optional[int]:
    """data pointer of a torch tensor / numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


PER_DEFAULTS = {"alpha": 0.6, "beta": 0.4, "beta_steps": 0, "eps": 1e-6}


def per_config(config: dict) -> Optional[dict]:
    """``buffer.prioritized`` of a YAML config, validated and completed with the defaults; None when absent or null (uniform
    sampling). Needs no device. ValueError for a bad range or a combination prioritized replay does not support."""
    p = (config.get("buffer") or {}).get("prioritized")
    if p is None:
        return None
    if not isinstance(p, dict):
        raise ValueError("buffer.prioritized must be a mapping {alpha, beta, beta_steps, eps} or null")
    unknown = set(p) - set(PER_DEFAULTS)
    if unknown:
        raise ValueError(f"buffer.prioritized: unknown keys {sorted(unknown)}")
    out = dict(PER_DEFAULTS, **p)
    alpha, beta, beta_steps, eps = float(out["alpha"]), float(out["beta"]), out["beta_steps"], float(out["eps"])
    if not alpha >= 0.0 or alpha != alpha or alpha == float("inf"):
        raise ValueError("buffer.prioritized.alpha must be a finite number >= 0")
    if not 0.0 <= beta <= 1.0:
        raise ValueError("buffer.prioritized.beta must be in [0, 1]")
    if isinstance(beta_steps, bool) or int(beta_steps) != beta_steps or int(beta_steps) < 0:
        raise ValueError("buffer.prioritized.beta_steps must be an integer >= 0")
    if not eps > 0.0 or eps == float("inf"):
        raise ValueError("buffer.prioritized.eps must be a finite number > 0")
    if (config.get("train") or {}).get("rng", "device") == "host":
        raise ValueError("buffer.prioritized needs train.rng: device (the tree samples on the device)")
    return {"alpha": alpha, "beta": beta, "beta_steps": int(beta_steps), "eps": eps}


def make_config(obs_dim: int, act_dim: int, config: dict, n_agents: int = 1, ctas_per_agent: int = 0,
                dp_world: int = 1, dp_rank: int = 0, batch_size: Optional[int] = None, agent_id_base: int = 0) -> SacxConfig:
    """YAML dict (reference: configs/example_config_env.yaml, sac/agent.py:22-115) -> sacx_config."""
    sac, qn, pn, tr = config["sac"], config["q_net"], config["policy_net"], config["train"]
    c = SacxConfig()
    c.obs_dim, c.act_dim = int(obs_dim), int(act_dim)
    ph, qh = list(pn["hidden_sizes"]), list(qn["hidden_sizes"])
    if not ph or not qh:
        raise ValueError("hidden_sizes cannot be empty")             # sac/models.py:135-136
    if len(ph) > SACX_MAX_HIDDEN or len(qh) > SACX_MAX_HIDDEN:
        raise ValueError(f"at most {SACX_MAX_HIDDEN} hidden layers are supported")
    c.n_hidden_pi, c.n_hidden_q = len(ph), len(qh)
    for i, h in enumerate(ph):
        c.hidden_pi[i] = int(h)
    for i, h in enumerate(qh):
        c.hidden_q[i] = int(h)
    # unknown names raise KeyError exactly like _ACTIVATIONS[...] in sac/models.py:138-139
    c.act_hidden_pi = ACTIVATION_IDS[pn["hidden_layers_act"]]
    c.act_out_pi = ACTIVATION_IDS[pn["output_activation"]]
    c.act_hidden_q = ACTIVATION_IDS[qn["hidden_layers_act"]]
    c.act_out_q = ACTIVATION_IDS[qn["output_activation"]]
    c.batch_size = int(batch_size if batch_size is not None else tr["batch_size"])
    c.auto_entropy_tuning = 1 if sac["auto_entropy_tuning"] else 0
    c.n_agents, c.ctas_per_agent = int(n_agents), int(ctas_per_agent)
    c.gamma, c.tau = float(sac["gamma"]), float(sac["tau"])
    c.log_std_min, c.log_std_max = float(pn["log_std_min"]), float(pn["log_std_max"])
    c.action_scale = float(pn["action_scale"])
    c.alpha = float(sac["alpha"])
    c.actor_lr, c.critic_lr, c.alpha_lr = float(sac["actor_lr"]), float(sac["critic_lr"]), float(sac["alpha_lr"])
    c.seed = int(tr.get("seed", 0)) & 0xFFFFFFFFFFFFFFFF
    c.dp_world, c.dp_rank = int(dp_world), int(dp_rank)
    c.agent_id_base = int(agent_id_base)
    return c
