"""Worker of tests/test_gpu_pbt_dist.py: one process per GPU (torchrun), the exploit step of population-based training over
REAL ranks. Local and cross-rank pairs (pack, one NCCL all_to_all_single, unpack) give every agent the bits the same exploit
gives an unsharded population in the same process, and so do three updates after it."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-actor-critic_b200"), HERE]

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from gpu_helpers import base_config
    from helpers import synth_transitions
    from sac.population import SACPopulation
    obs, act, B, n = 4, 1, 64, 4 * world + 1
    cfg = base_config(hidden=(32, 32), batch=B, capacity=2000, rng="device", auto=False)
    seeds = [5 + g for g in range(n)]
    trials = [{"alpha": 0.05 + 0.01 * g, "actor_lr": 1e-4 * (1 + g), "tau": 0.001 * (1 + g)} for g in range(n)]
    s, a, r, s2, d = (torch.from_numpy(x).cuda() for x in synth_transitions(1500, obs, act, 3))
    pops = {}
    for name, kw in (("sharded", {}), ("whole", {"rank": 0, "world": 1})):
        pop = SACPopulation(obs, act, cfg, n, seeds=seeds, reference_init=False, **kw)
        if name == "whole":                 # the sharded initialisation draws one stream per rank: give the whole the same weights
            for q in range(world):
                from sac.population import shard_agents
                ids = list(shard_agents(n, world, q))
                src = torch.empty((len(ids), pops["sharded"].engine.stride), device="cuda")
                if q == rank:
                    src.copy_(pops["sharded"].engine.arena.view(len(ids), -1))
                dist.broadcast(src, q)
                pop.engine.arena.view(n, -1)[ids[0]: ids[-1] + 1].copy_(src)
        pop.push_device_all(s, a, r, s2, d.float())
        pop.set_trials(trials)
        pop.update(2)
        pops[name] = pop
    last = n - 1                            # pairs: cross-rank both ways, one source feeding several ranks, local pairs
    pairs = [(0, last), (0, 1), (last - 1, 2), (0, n // 2), (n // 2 + 1, n // 2 + 2)]
    hypers = [None, {"gamma": 0.97}, {"alpha": 0.11, "critic_lr": 4e-4}, {"tau": 0.03}, None]
    for pop in pops.values():
        pop.exploit(pairs, hypers)
    torch.cuda.synchronize()

    def check(what):
        sh, wh = pops["sharded"], pops["whole"]
        for a_loc, g in enumerate(sh.agent_ids):
            x = sh.engine.arena.view(torch.int32).view(sh.n_local, -1)[a_loc]
            y = wh.engine.arena.view(torch.int32).view(n, -1)[g]
            assert torch.equal(x, y), f"{what}: agent {g} differs from the unsharded population"

    check("after exploit")
    for pop in pops.values():
        pop.update(3)
    torch.cuda.synchronize()
    check("after 3 updates")
    dist.barrier()
    if rank == 0:
        print(f"DIST_OK pbt world={world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
