"""Cost of n-step returns (buffer.n_step) per update: python tools/nstep_bench.py [--rounds R] [--out FILE]

For each workload of bench.py that selects a different update path -- bipedal (row-parallel kernel, BipedalWalker shape,
batch 256, 1M-slot ring, device RNG), donkey (FFMA tiles, batch 1024) and population (1024 agents, tensor-core path) --
one engine per n in (1, 3, 5, 10) is built in this process on the same seeded ring, and the engines are timed in alternation
for R rounds (CUDA events around a device-resident burst of updates, after a warm-up). Prints ONE JSON line: the card's name
and power limit read in the same run, and per workload and n the median / min / max updates per second (agent-updates for
the population) over the rounds, and the median overhead against n = 1."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-actor-critic_b200")]

NS = (1, 3, 5, 10)
# workload: (updates per timed burst = per launch, warm-up updates)
PLAN = {"bipedal": (1000, 200), "donkey": (400, 50), "population": (20, 3)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, mhz = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit_w": float(pl), "sm_max_mhz": float(mhz)}
    except Exception as ex:                                   # the card name still comes from the driver
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "error": str(ex)}


def build(name, n):
    import torch
    import bench
    w = dict(bench.WORKLOADS[name])
    cfg = bench.make_config(w, "device", seed=0)
    cfg["buffer"]["n_step"] = n
    s, a, r, s2, d = bench.synth(w["fill"], w["obs"], w["act"], seed=0)
    if w["n_agents"] == 1:
        from sac.agent import SAC
        agent = SAC(bench.FakeEnv(w["obs"], w["act"]), cfg)
        agent.replay_buffer.push_batch(s, a, r, s2, d)
        eng, keep = agent.engine, agent
    else:
        from sac.population import SACPopulation
        pop = SACPopulation(w["obs"], w["act"], cfg, w["n_agents"], rank=0, world=1, reference_init=False)
        pop.push_device_all(*(torch.from_numpy(x).cuda() for x in (s, a, r, s2, d)))
        eng, keep = pop.engine, pop
    torch.cuda.synchronize()
    return eng, keep, w["n_agents"]


def time_burst(eng, k):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    eng.update(None, None, None, k)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--workloads", default=",".join(PLAN))
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nstep_bench.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    res = {"card": card(), "rounds": args.rounds, "n_step": list(NS), "workloads": {}}
    for name in args.workloads.split(","):
        k, warm = PLAN[name]
        engines = {n: build(name, n) for n in NS}
        path = engines[1][0].path()[0] + ("+tensor-core" if engines[1][0].tensor_core()[0] else "")
        for n in NS:
            engines[n][0].update(None, None, None, warm)
        rates = {n: [] for n in NS}
        for rnd in range(args.rounds):
            order = NS if rnd % 2 == 0 else NS[::-1]           # alternate the order: no n always runs first
            for n in order:
                eng, _, agents = engines[n]
                rates[n].append(k * agents / time_burst(eng, k))
        med = {n: float(np.median(rates[n])) for n in NS}
        res["workloads"][name] = {
            "path": path, "updates_per_launch": k,
            "unit": "agent-updates/s" if engines[1][2] > 1 else "updates/s",
            "rates": {str(n): {"median": med[n], "min": float(min(rates[n])), "max": float(max(rates[n]))} for n in NS},
            "overhead_pct_vs_n1": {str(n): 100.0 * (med[1] / med[n] - 1.0) for n in NS if n > 1},
            "us_per_update": {str(n): 1e6 * engines[n][2] / med[n] for n in NS},
        }
        del engines
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
