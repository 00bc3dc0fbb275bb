#!/usr/bin/env python
"""bench.py -- SAC updates/s at BipedalWalker shape (BASELINE.json configs[1]) on N B200s.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload bipedal|population|donkey|dp] [--no-extras]
                    [--dump-outputs DIR]

A "step" is one full SAC gradient update (ring gather + target + 2 critic steps + actor step + temperature step
+ Polyak; reference: SAC.training_step, sac/agent.py:302-327) on synthetic transitions (SURVEY section 8d).
One JSON line is printed by rank 0:
  value     updates/s with everything resident in HBM (device RNG, K updates timed with CUDA events)
  e2e       updates/s through the public API SAC.training_step() in host-RNG mode: every step draws the
            reference's index stream + normals on the host, copies them from pinned memory (H2D), runs the
            fused kernel and reads the metrics back (D2H)
  roofline  the fused update kernel against the measured peaks (MEASURED_PEAKS.json)
  cpu_baseline  the torch-eager CPU port of the reference (oracle/torch_port.py) on this box's host cores
N > 1: the single-agent update does not shard ("replicas only", DESIGN.md): every rank runs an independent
agent (the population-of-seeds mode, no collective on the data path); value = all ranks' updates / max time.
The two modes that DO shard ride along in `extra` of the same line (default workload only): `extra.population` --
1024 InvertedPendulum-shape agents with 100000-row rings partitioned over the ranks, no collective -- and `extra.dp` --
BipedalWalker shape at global batch 65536 split over the ranks, two NCCL all-reduces per update, with the in-run checks
that the replicas stay bit-identical and within 2e-5 of the single-rank result, and the all-reduce share of the update.
Timing: W warm-up steps, then exactly K timed steps in up to 5 repeats of near-equal length; the median repeat's time per
step is reported.
--dump-outputs DIR: after the timed steps, what the timed path computed in its last step goes to DIR/<name>.npy (see
dump_outputs). The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "soft-actor-critic_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (obs, act, hidden, batch, ring capacity, fill, n_agents, activation)
    "bipedal": dict(obs=24, act=4, hidden=[256, 256], batch=256, capacity=1_000_000, fill=1_000_000, n_agents=1, act_fn="relu",
                    label="BipedalWalker-v3 shape: obs 24, act 4, 2x256 relu MLPs, batch 256, 1M-transition ring (216 MB > L2)"),
    "donkey": dict(obs=32, act=2, hidden=[256, 256], batch=1024, capacity=50_000, fill=50_000, n_agents=1, act_fn="relu",
                   label="DonkeyVae latent shape: obs 32, act 2, 2x256 relu, batch 1024, 50k ring"),
    "population": dict(obs=4, act=1, hidden=[256, 256], batch=256, capacity=100_000, fill=100_000, n_agents=1024, act_fn="relu",
                       label="InvertedPendulum shape: obs 4, act 1, 2x256, batch 256, 1024 independent agents sharded over ranks"),
    "dp": dict(obs=24, act=4, hidden=[256, 256], batch=65536, capacity=1_000_000, fill=1_000_000, n_agents=1, act_fn="relu", dp=True,
               label="large-batch data parallel: BipedalWalker shape, global batch 65536 split over ranks, 2 NCCL all-reduces per update"),
}


def flops_per_update(obs, act, hidden, batch):
    """Algorithmic FLOPs of one update (SURVEY section 8a): 2*MACs, no autograd waste."""
    dims_p = [obs] + hidden + [2 * act]
    dims_q = [obs + act] + hidden + [1]
    FP = sum(a * b for a, b in zip(dims_p[:-1], dims_p[1:]))
    FQ = sum(a * b for a, b in zip(dims_q[:-1], dims_q[1:]))
    macs = 2 * FP + 6 * FQ + 2 * (2 * FQ - (obs + act) * hidden[0]) + 2 * (FQ - obs * hidden[0]) + (2 * FP - obs * hidden[0])
    return 2 * macs * batch


def param_counts(obs, act, hidden):
    dims_p = [obs] + hidden + [2 * act]
    dims_q = [obs + act] + hidden + [1]
    NP = sum(a * b + b for a, b in zip(dims_p[:-1], dims_p[1:]))
    NQ = sum(a * b + b for a, b in zip(dims_q[:-1], dims_q[1:]))
    return NP + 2 * NQ, 2 * NQ


def bytes_per_update(obs, act, hidden, batch):
    """Algorithmic bytes (SURVEY section 8d): gather + read theta,theta_bar + r/w m,v + write theta, theta_bar."""
    n_on, n_tg = param_counts(obs, act, hidden)
    return batch * (2 * obs + act + 2) * 4 + 4 * (n_on + n_tg) + 16 * n_on + 4 * n_on + 4 * n_tg


def make_config(w, rng, seed=0):
    return {
        "sac": {"gamma": 0.99, "tau": 0.005, "alpha": 0.1, "auto_entropy_tuning": True,
                "actor_lr": 3e-4, "critic_lr": 3e-4, "alpha_lr": 3e-4},
        "q_net": {"hidden_sizes": list(w["hidden"]), "hidden_layers_act": w["act_fn"], "output_activation": "identity"},
        "policy_net": {"hidden_sizes": list(w["hidden"]), "hidden_layers_act": w["act_fn"], "output_activation": "identity",
                       "log_std_min": -20, "log_std_max": 2, "action_scale": 1.0},
        "buffer": {"capacity": w["capacity"]},
        "train": {"gradient_steps_per_update": 1, "seed": seed, "batch_size": w["batch"], "warming_steps": 1000,
                  "device": "cuda", "rng": rng},
        "logger": {"enabled": False, "log_dir": "runs", "env_name": "Synthetic", "agent_name": "SAC", "run_name": "bench",
                   "use_timestamp": False, "timestamp_format": "%Y", "flush_secs": 10, "log_episode_stats": False,
                   "log_q_values": False, "save_model": {"enabled": False, "path": None}},
    }


def synth(n, obs, act, seed=0):
    rng = np.random.default_rng(seed)
    s = rng.standard_normal((n, obs), dtype=np.float32)
    s2 = rng.standard_normal((n, obs), dtype=np.float32)
    a = rng.uniform(-1, 1, (n, act)).astype(np.float32)
    r = rng.standard_normal(n, dtype=np.float32)
    d = (rng.random(n) < 0.01).astype(np.float32)
    return s, a, r, s2, d


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class _Space:
    def __init__(self, n):
        self.shape = (n,)

    def seed(self, s):
        return [s]


class FakeEnv:
    """Shape-only environment: the benchmark feeds synthetic transitions, no simulator."""
    spec = None

    def __init__(self, obs, act):
        self.observation_space, self.action_space = _Space(obs), _Space(act)

    def reset(self, seed=None):
        return np.zeros(self.observation_space.shape, np.float32), {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU baseline
def cpu_reference(w, steps, warmup, budget_s=40.0, fill_cap=None):
    """The reference's CPU update (torch-eager port, pinned bit-exact to the reference in tests/) on this box's
    host cores. Comparator (A): full training_step incl. random.sample on the filled deque; (B): compute only."""
    import torch
    from oracle.torch_port import TorchPortSAC

    cfg = make_config(w, "host")
    cfg["train"]["device"] = "cpu"
    port = TorchPortSAC(w["obs"], w["act"], cfg, capacity=w["capacity"])
    n = w["fill"] if fill_cap is None else min(w["fill"], fill_cap)
    s, a, r, s2, d = synth(n, w["obs"], w["act"])
    t0 = time.perf_counter()
    rl, dl = r.tolist(), (d != 0).tolist()
    for i in range(n):
        port.push(s[i], a[i], rl[i], s2[i], dl[i])
    fill_s = time.perf_counter() - t0
    nproc = os.cpu_count() or 1
    best = None
    for threads in sorted({1, max(1, nproc // 2), nproc}):
        torch.set_num_threads(threads)
        for _ in range(max(3, min(warmup, 10))):
            port.training_step()
        k, t0 = 0, time.perf_counter()
        while k < steps and (time.perf_counter() - t0) < budget_s / 3:
            port.training_step()
            k += 1
        dt = time.perf_counter() - t0
        if best is None or k / dt > best["value"]:
            best = {"value": k / dt, "cores": threads, "updates": k, "seconds": dt}
    torch.set_num_threads(best["cores"])
    batch = port.sample_batch(w["batch"])
    for _ in range(3):
        port.update_from_batch(*batch)
    k, t0 = 0, time.perf_counter()
    while k < steps and (time.perf_counter() - t0) < budget_s / 4:
        port.update_from_batch(*batch)
        k += 1
    compute_only = k / (time.perf_counter() - t0)
    return {"value": best["value"], "unit": "updates/s", "cores": best["cores"], "host_cores": nproc, "kind": "port", "updates": best["updates"],
            "sample": f"{best['updates']} full training_step() calls (deque of {n} transitions, random.sample + eager torch + Adam) in {best['seconds']:.1f}s; "
                      f"thread sweep {{1,{max(1, nproc // 2)},{nproc}}}, best kept",
            "compute_only_value": compute_only, "fill_seconds": fill_s}


# ---------------------------------------------------------------------------------------------- measurement
L2_NOTE = {
    "bipedal": "inputs larger than L2: 216 MB ring, every update gathers 256 fresh random rows (no flush needed)",
    "donkey": "L2-resident by nature: 10.8 MB ring + 9 MB arena fit the 126 MB L2 (as they would in production); no flush",
    "population": "inputs larger than L2: {agents} agents x (4.4 MB ring + 9 MB arena) = {gb:.1f} GB streamed per sweep",
    "dp": "inputs larger than L2: 216 MB ring, 65536 random rows per update, ~0.9 GB of activations per rank",
}


class Runner:
    """One workload on this rank: engine + ring, a `run(n)` that performs n steps on the current stream."""

    def __init__(self, name, rank, world, chunk):
        import torch
        self.name, self.rank, self.world, self.chunk = name, rank, world, chunk
        w = self.w = WORKLOADS[name]
        self.agent = self.dp = self.pop = None
        self.scaling = "weak"
        if w.get("dp"):
            from sac.population import DataParallelSAC
            self.scaling = "strong"
            self.dp = DataParallelSAC(w["obs"], w["act"], make_config(w, "device", seed=0), w["batch"], rank=rank, world=world)
            self.eng, self.ring = self.dp.engine, self.dp.ring
            self.ring.push_batch(*synth(w["fill"], w["obs"], w["act"], seed=0))          # ring replicated on every rank
            self.n_local = 1
        elif w["n_agents"] == 1:
            from sac.agent import SAC
            self.agent = SAC(FakeEnv(w["obs"], w["act"]), make_config(w, "device", seed=rank))
            self.eng, self.ring = self.agent.engine, self.agent.replay_buffer
            self.ring.push_batch(*synth(w["fill"], w["obs"], w["act"], seed=rank))
            self.n_local = 1
        else:
            from sac.population import SACPopulation
            self.scaling = "strong"                                   # 1024 agents in total, partitioned over the ranks
            self.pop = SACPopulation(w["obs"], w["act"], make_config(w, "device", seed=0), w["n_agents"], rank=rank, world=world,
                                     reference_init=False)
            self.eng, self.ring, self.n_local = self.pop.engine, self.pop.ring, self.pop.n_local
            s, a, r, s2, d = synth(w["fill"], w["obs"], w["act"], seed=rank)
            self.pop.push_device_all(*(torch.from_numpy(x).cuda() for x in (s, a, r, s2, d)))
        torch.cuda.synchronize()

    def run(self, n):
        if self.dp is not None:
            for _ in range(n):
                self.dp.update()
            return
        done = 0
        while done < n:
            c = min(self.chunk, n - done)
            self.eng.update(None, None, None, c)
            done += c

    def units(self, steps):
        """work units (updates / agent-updates) ALL ranks complete in `steps` steps"""
        w = self.w
        if self.dp is not None:
            return steps                                             # one global-batch update per step, whatever G is
        if w["n_agents"] > 1:
            return steps * w["n_agents"]                             # every agent of the population, wherever it lives
        return steps * self.world                                    # replicas: one independent agent per rank


def timed(runner, steps, warmup, barrier, dist, world, max_repeats=5):
    """W warm-up steps, then EXACTLY `steps` steps split into min(5, steps) repeats of near-equal length, each repeat bracketed
    by barrier + synchronize on both sides and timed with CUDA events on the launching stream; per repeat the MAX over ranks.
    Returns the MEDIAN repeat's ms per step and every repeat's (steps, ms)."""
    import torch
    runner.run(warmup)
    barrier()
    n = min(max_repeats, steps)
    reps = []
    for k in [steps // n + (i < steps % n) for i in range(n)]:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        runner.run(k)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        reps.append((k, ms))
    return float(np.median([ms / k for k, ms in reps])), reps


DUMP_TENSORS = re.compile(r"(pi|q1|q2|q1t|q2t)\.[Wb]\d+|out\.(y|logpi|q1|q2)|scal\.(log_alpha|alpha)")


def dump_outputs(runner, out_dir, max_agents=16, max_bytes=64 << 20):
    """What the last update left for its caller, one DIR/<name>.npy per array: every network's weights and biases (pi, q1, q2)
    and the target copies (q1t, q2t) as float32, the temperature (scal.alpha, scal.log_alpha) as float64, the per-row outputs
    of the batch (out.y Bellman target, out.logpi, out.q1, out.q2) and the update's metrics (metrics.<key>, float64).
    A population writes a fixed, seeded sample of `max_agents` of this rank's agents, stacked on a leading axis."""
    import torch
    eng = runner.eng
    torch.cuda.synchronize()
    agents = [0]
    if eng.n_agents > 1:
        agents = sorted(np.random.default_rng(0).choice(eng.n_agents, min(max_agents, eng.n_agents), replace=False).tolist())

    def stack(vals):
        return vals[0] if eng.n_agents == 1 else np.stack(vals)

    arrays = {name: stack([eng.view(name, a).cpu().numpy() for a in agents]) for name in eng.layout if DUMP_TENSORS.fullmatch(name)}
    if eng.n_agents > 1:
        arrays["agents"] = np.asarray(agents, np.float64)
    metrics = [eng.metrics(a) for a in agents]
    for key in metrics[0]:
        arrays[f"metrics.{key}"] = stack([np.float64(m[key]) for m in metrics])
    total = sum(v.nbytes for v in arrays.values())
    assert total <= max_bytes, f"output dump of {total} bytes exceeds {max_bytes}"
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(v))


def dp_checks(runner, dist, world, rank):
    """In-run parity of the data-parallel mode (SURVEY cfg 5): after 3 updates the replicated parameters are bit-identical on
    every rank, and within 2e-5 rel-L2 of the SAME 3 updates done by one rank on the whole 65536-row batch (device RNG is
    keyed by the global row, so the global batch does not depend on G)."""
    import torch
    from sac.population import DataParallelSAC
    w = runner.w
    for _ in range(3):
        runner.dp.update()
    torch.cuda.synchronize()
    p = runner.eng.view("block.params").reshape(-1).clone()
    out = {"ranks_bit_identical": True, "vs_single_rank_rel_l2": 0.0}
    if world > 1:
        hi, lo = p.clone(), p.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        out["ranks_bit_identical"] = bool(torch.equal(hi, lo))
        assert out["ranks_bit_identical"], "data-parallel replicas diverged"
        if rank == 0:
            one = DataParallelSAC(w["obs"], w["act"], make_config(w, "device", seed=0), w["batch"], rank=0, world=1)
            one.ring.push_batch(*synth(w["fill"], w["obs"], w["act"], seed=0))
            for _ in range(3):
                one.update()
            torch.cuda.synchronize()
            q = one.engine.view("block.params").reshape(-1)
            out["vs_single_rank_rel_l2"] = float((p.double() - q.double()).norm() / q.double().norm())
            assert out["vs_single_rank_rel_l2"] < 2e-5, out
            del one
            torch.cuda.empty_cache()
        dist.barrier()
    return out


def measure(name, args, rank, world, local_rank, barrier, dist, steps, warmup, with_clocks, dump_dir=None):
    import torch
    runner = Runner(name, rank, world, args.chunk)
    w, eng = runner.w, runner.eng
    extra = {}
    if runner.dp is not None:
        extra["parity"] = dp_checks(runner, dist, world, rank)
    clocks = None
    if with_clocks:
        clocks = ClockSampler(local_rank)
        clocks.start()
    l0 = eng.launch_count()
    ms, reps = timed(runner, steps, warmup, barrier, dist, world)
    launches = eng.launch_count() - l0
    if dump_dir and rank == 0:                                       # before anything below runs more updates
        dump_outputs(runner, dump_dir)
    if runner.dp is not None and world > 1:                           # share of the update spent inside the two all-reduces
        runner.dp.time_exchange = True
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        runner.run(steps)
        ev1.record()
        torch.cuda.synchronize()
        xms = runner.dp.exchange_ms()
        runner.dp.time_exchange = False
        extra["allreduce_ms_per_update"] = xms / steps
        extra["allreduce_share"] = xms / ev0.elapsed_time(ev1)
        extra["exchange"] = "two ncclAllReduce per update on the engine stream: 588 KB critic gradients; 297 KB policy gradients + temperature share"
        extra["limiter"] = ("the two all-reduces" if extra["allreduce_share"] > 0.25 else
                            "not the exchange: per-update fixed cost that does not shrink with the per-rank batch (about 38 launches per "
                            "update and the parameter-sized passes: dW split reduction, Adam, Polyak)")
    clk = None
    if clocks is not None:
        if sum(t for _, t in reps) < 1500:                           # a longer stretch for the clock sampler (outside the timed region)
            runner.run(int(min(50000, 1500 / max(ms, 1e-3))))
            torch.cuda.synchronize()
        clk = clocks.stop()
    m = eng.metrics()
    assert m["nonfinite"] == 0 and np.isfinite(m["q1_loss"]), f"non-finite update: {m}"
    value = runner.units(1) / (ms / 1000.0)
    tc_on, _, tc_launches = eng.tensor_core()
    path = "tensor-core" if tc_on else eng.path()[0]
    gx, gy, smem = eng.grid()
    per_step = [t / k for k, t in reps]
    res = {"value": value, "unit": "agent-updates/s" if w["n_agents"] > 1 else "updates/s", "ms_per_step": ms, "steps": steps,
           "repeats": len(reps), "ms_per_step_min": min(per_step), "ms_per_step_max": max(per_step), "scaling": runner.scaling,
           "path": path, "gpu_launches_per_step": launches / steps, "agents_per_gpu": runner.n_local,
           "workload": w["label"], "grid": [gx, gy], "smem_bytes": smem, "tc_kernel_launches": int(tc_launches),
           "l2": L2_NOTE[name].format(agents=runner.n_local, gb=runner.n_local * (w["fill"] * (2 * w["obs"] + w["act"] + 2) * 4 + 9.0e6) / 1e9),
           "final_metrics": {k: m[k] for k in ("q1_loss", "policy_loss", "alpha", "updates")}, **extra}
    return runner, res, clk, launches


def roofline_of(name, res, world, pk):
    w = WORKLOADS[name]
    fl = flops_per_update(w["obs"], w["act"], w["hidden"], w["batch"])
    by = bytes_per_update(w["obs"], w["act"], w["hidden"], w["batch"])
    per_gpu_rate = res["value"] / world                               # (agent-)updates/s on one GPU
    if w.get("dp"):
        fl, per_gpu_rate = fl // world, res["value"]                  # per rank: 1/G of the batch FLOPs; every rank joins every update
    ach_tf = fl * per_gpu_rate / 1e12
    traffic, traffic_note = None, None
    prof = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                ent = json.load(f).get(name, {})
            traffic, traffic_note = ent.get("dram_bytes_per_update"), ent.get("dram_bytes_note")
        except Exception:
            pass
    if res["path"] == "tensor-core":
        kernel = ("sacx_tc_kernel (tcgen05 3xTF32 tiles, TMEM accumulators, TMA operands) + sacx_rows_kernel + tc_dw_reduce_kernel; "
                  "achieved = algorithmic FLOP of the whole update / measured time per update (profiles/: per-kernel launch list)")
        note = ("every product is three TF32 MMAs (hi/lo split, fp32-level accuracy: parity contract rel 1e-4), so the ceiling of this "
                "path is one third of the TF32 rate, about one sixth of the bf16 peak the fraction is quoted against")
    elif res["path"] == "rowpar":
        kernel = "sacx_rp_kernel (persistent row-parallel fused update: 3xTF32 mma.sync tiles, 4 grid barriers per update)"
        note = "single agent at batch 256 is latency-bound (dependent 16-row GEMM jobs, group + grid barriers): see profiles/ (phase trace)"
    else:
        kernel = "sacx_run_kernel (persistent tile-parallel fused update, FP32 FFMA tiles)"
        note = "FP32 FFMA path; one grid barrier per dependent layer"
    return {"bound": "tensor", "achieved": ach_tf, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": ach_tf / pk["bf16_tflops_sustained"], "traffic": traffic, "traffic_note": traffic_note,
            "kernel": kernel, "peak_source": pk["source"] + ", sustained bf16 (kernel timed inside a long loop)",
            "flop_per_update": fl, "fp32_ffma_nominal_tflops": 148 * 128 * 2 * 1.965e-3,
            "frac_of_fp32_ffma_nominal": ach_tf / (148 * 128 * 2 * 1.965e-3),
            "hbm_view": {"bytes_per_update": by, "achieved_gbs": by * per_gpu_rate / 1e9, "peak_gbs": pk["hbm_gbs"],
                         "frac": by * per_gpu_rate / 1e9 / pk["hbm_gbs"]},
            "note": note}


def e2e_through_public_api(agent, w, args, W, world, barrier, dist):
    """The same metric through the call a user makes -- SAC.training_step() in host-RNG mode: every step draws the reference's
    index stream (random.sample) and normals (torch CPU generator) on the host, copies them from pinned memory (H2D), runs the
    fused kernel and copies the step's metrics block back (D2H). last_metrics() at the end waits for the last step."""
    import random
    import torch
    agent.rng_mode = "host"
    random.seed(0)
    torch.manual_seed(0)
    B, A = w["batch"], w["act"]
    n = args.e2e_steps or max(min(args.steps, 2000), 200)
    for _ in range(max(3, min(W, 50))):
        agent.training_step()
    agent.last_metrics()
    reps = []
    while len(reps) < 5 or (sum(reps) < 500.0 and len(reps) < 50):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(n):
            agent.training_step()
        mm = agent.last_metrics()
        e1.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1000.0
        assert mm["nonfinite"] == 0 and np.isfinite(mm["q1_loss"])
        ms = max(e0.elapsed_time(e1), wall - 1.0)          # (the event pair cannot see host time before the first enqueue)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        reps.append(ms)
    ms = float(np.median(reps))
    return {"value": n * world / (ms / 1000.0), "unit": "updates/s", "h2d_bytes_per_step": B * 8 + 2 * B * A * 4,
            "d2h_bytes_per_step": 232, "steps": n, "repeats": len(reps), "ms_per_step": ms / n,
            "api": "SAC.training_step() with train.rng = 'host' (random.sample index stream + torch CPU normals -> pinned H2D -> fused "
                   "kernel -> metrics D2H), then SAC.last_metrics(); median of the repeats"}


# ---------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bipedal", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the population / data-parallel legs of the default run")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = clamp(steps, 200, 2000)")
    ap.add_argument("--chunk", type=int, default=1000, help="updates per kernel launch in the device-resident loop")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    W = max(3, args.warmup)

    if args.impl == "reference":
        if rank != 0:
            return
        steps = min(args.steps, 600)
        base = cpu_reference(w, steps, W, budget_s=120.0)
        line = {"impl": "reference", "metric": "SAC updates/s", "value": base["value"], "unit": "updates/s", "n_gpus": args.gpus,
                "steps": base["updates"], "warmup": W,
                "ms_per_step": 1000.0 / base["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": {"workload": w["label"], "device": "host CPU"},
                "cpu_baseline": base, "e2e": {"value": base["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the update path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- headline workload: device-resident throughput, then the same metric through the public API -----------------------
    runner, res, clk, launches = measure(args.workload, args, rank, world, local_rank, barrier, dist, args.steps, W, True,
                                         args.dump_outputs)
    e2e = None
    if runner.agent is not None:
        e2e = e2e_through_public_api(runner.agent, w, args, W, world, barrier, dist)
    del runner
    torch.cuda.empty_cache()

    # ---- the modes that SHARD (SURVEY 8e), attached to the same line so that the driver's 1/2/4/8 runs record their curves:
    # population of 1024 agents partitioned over the ranks (no collective); global batch 65536 split over the ranks (2 all-reduces)
    extras = {}
    if args.workload == "bipedal" and not args.no_extras:
        for name, k, wu in (("population", 60, 3), ("dp", 250, 10)):          # about 0.5 s timed each on one B200
            r2, x, _, _ = measure(name, args, rank, world, local_rank, barrier, dist, k, wu, False)
            del r2
            torch.cuda.empty_cache()
            extras[name] = x

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    roofline = roofline_of(args.workload, res, world, pk)
    for name, x in extras.items():
        rf = roofline_of(name, x, world, pk)
        x["roofline"] = {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "hbm_view", "flop_per_update")}
        x["n_gpus"] = world
    cpu = None
    if not args.no_cpu_baseline and world == 1:          # (the contract: timed on rank 0 at N=1 only)
        cpu = cpu_reference(w if w["n_agents"] == 1 else dict(w, fill=w["fill"]), 400, 10, budget_s=40.0)
    line = {"metric": "SAC updates/s", "value": res["value"], "unit": "updates/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": res["ms_per_step"], "repeats": res["repeats"], "ms_per_step_min": res["ms_per_step_min"],
            "ms_per_step_max": res["ms_per_step_max"], "higher_is_better": True, "scaling": res["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["label"], "agents_per_gpu": res["agents_per_gpu"], "updates_per_launch": args.chunk, "l2": res["l2"],
                       "grid": res["grid"], "smem_bytes": res["smem_bytes"], "path": res["path"], "tc_kernel_launches": res["tc_kernel_launches"],
                       "timing": "median of the repeats; each repeat = `steps` updates between barrier+synchronize, CUDA events, max over ranks",
                       "multi_gpu": ("data parallel: 2 NCCL all-reduces per update" if w.get("dp") else
                                     "population sharded over ranks, no collective" if w["n_agents"] > 1 else
                                     "replicas only (independent agents per rank, no collective); the sharded modes are in `extra`")},
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "final_metrics": res["final_metrics"], "extra": extras}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
