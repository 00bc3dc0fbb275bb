"""Cost of one exploit round of population-based training at bench.py's population workload (1024 agents, obs 4 / act 1 /
2x256, batch 256, 100 000-row rings): 204 (source, destination) pairs with hyper-parameter records, i.e. fraction 0.2.

    python tools/pbt_bench.py [--reps 20] [--out FILE]                                 # one GPU: every pair is a local copy
    python -m torch.distributed.run --nproc-per-node=N tools/pbt_bench.py [...]       # N ranks: every pair crosses ranks

Per round: time from CUDA events around SACPopulation.exploit, host work included (median of --reps rounds, max over
ranks); on one GPU also the copy launch alone, 20 rounds queued back to back; the learner
state's size from the arena layout (sacx_pbt_state_floats, not measured), bytes/s against the HBM copy peak the project measured
(6.55 TB/s, DESIGN.md section 4), and the round's share of an interval of 1 000 update sweeps timed in the same process. The
card's name and power limit are read in the same run. Writes nothing unless --out is given."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-actor-critic_b200")]

import numpy as np  # noqa: E402

COPY_PEAK_TBS = 6.55


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sweeps", type=int, default=20, help="update sweeps timed for the interval share")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from bench import Runner, WORKLOADS
    w = WORKLOADS["population"]
    runner = Runner("population", rank, world, chunk=10)
    pop, eng = runner.pop, runner.eng
    n = w["n_agents"]
    k = int(0.2 * n)
    pairs = [(n - 1 - i, i) for i in range(k)]                    # top 204 -> bottom 204: all local on 1 rank, all cross-rank on N
    hypers = [{"alpha_lr": 3e-4 * (1 + 1e-3 * i), "actor_lr": 3e-4 * (1 - 1e-3 * i), "critic_lr": 2e-4 * (1 + 1e-3 * i),
               "tau": 0.005 * (1 + 1e-3 * i), "gamma": 0.99} for i in range(k)]
    state_bytes = 4 * eng.pbt_state_floats()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(3):
        pop.exploit(pairs, hypers)
    ms = []
    for _ in range(args.reps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pop.exploit(pairs, hypers)
        e1.record()
        barrier()
        ms.append(max_over_ranks(e0.elapsed_time(e1)))
    round_ms = float(np.median(ms))
    # device time alone: the same round's launches queued back to back (records and routes built once, outside the window)
    from sac.pbt import pbt_record, route_exploit
    rt = route_exploit(pairs, n, world)[rank]
    recs = [pbt_record(h, bool(pop.config["sac"]["auto_entropy_tuning"])) for h in hypers]
    queued_ms = None
    if world == 1:
        b2b = 20
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(b2b):
            eng.pbt_copy(rt.copy_src, rt.copy_dst, [recs[i] for i in rt.copy_pair])
        e1.record()
        barrier()
        queued_ms = e0.elapsed_time(e1) / b2b
    runner.run(5)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    runner.run(args.sweeps)
    e1.record()
    barrier()
    sweep_ms = max_over_ranks(e0.elapsed_time(e1)) / args.sweeps
    if rank == 0:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        cards = sorted(set(l.strip() for l in smi.stdout.strip().splitlines()[:world]))
        moved = 2 * k * state_bytes                                # each state read once and written once (local copy)
        res = {
            "workload": w["label"], "gpus": world, "cards": cards, "pairs": k, "records": True,
            "pairs_cross_rank": world > 1,
            "state_bytes_per_agent": state_bytes, "state_mb_per_agent": round(state_bytes / 1e6, 3),
            "round_ms_median": round(round_ms, 4), "round_ms_min": round(min(ms), 4), "round_ms_max": round(max(ms), 4),
            "states_delivered_gb_per_s": round(k * state_bytes / (round_ms * 1e-3) / 1e9, 1),
            "sweep_ms": round(sweep_ms, 4),
            "share_of_1000_sweeps": round(round_ms / (1000 * sweep_ms + round_ms), 6),
        }
        if world == 1:
            res["copy_ms_back_to_back"] = round(queued_ms, 4)
            res["copy_tb_per_s_back_to_back"] = round(moved / (queued_ms * 1e-3) / 1e12, 3)
            res["copy_tb_per_s_read_plus_write"] = round(moved / (round_ms * 1e-3) / 1e12, 3)
            res["share_of_copy_peak_back_to_back"] = round(res["copy_tb_per_s_back_to_back"] / COPY_PEAK_TBS, 3)
        line = json.dumps(res)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
