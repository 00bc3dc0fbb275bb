"""Prioritized replay cost on the GPU: python tools/per_bench.py [--out FILE] [--repeats R] [--updates N]

One JSON line (stdout, and FILE when given) with
  * the card's name and power limit (nvidia-smi, read in this run);
  * updates/s of the default workload (BipedalWalker shape: obs 24, act 4, 2 x 256, batch 256, 1M-slot ring), uniform sampling
    (device Feistel sampler, N updates per launch as bench.py runs them) and prioritized replay (buffer.prioritized), the two
    alternated R times in this process; median, min and max over the repeats;
  * CUDA-event times per call of the tree's sync + sample (sacx_per_sample) and of the priority write-back
    (sacx_per_update_priorities) on a 1M-leaf tree at B 256 and B 65 536;
  * kernel launches per prioritized update."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-actor-critic_b200"), os.path.join(ROOT, "tests")]

OBS, ACT, CAP, BATCH = 24, 4, 1 << 20, 256


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split("\n")[0].split(",")]
    return name, power


def fill(buf, n):
    g = torch.Generator(device="cuda").manual_seed(0)
    for i in range(0, n, 1 << 18):
        m = min(1 << 18, n - i)
        r = lambda *s: torch.randn(*s, device="cuda", generator=g)
        buf.push_device(r(m, OBS), r(m, ACT).clamp_(-1, 1), r(m), r(m, OBS), (torch.rand(m, device="cuda", generator=g) < 0.01).float())


def event_time(fn, n):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / n          # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--updates", type=int, default=2000)
    args = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    from gpu_helpers import base_config
    from sac import _engine as E
    from sac.engine import UpdateEngine
    from sac.replay_buffer import PrioritizedReplayBuffer, ReplayBuffer
    name, power = card()
    torch.cuda.set_device(0)

    cfg = base_config(hidden=(256, 256), batch=BATCH, capacity=CAP, rng="device")
    legs = {}
    for kind in ("uniform", "per"):
        if kind == "uniform":
            buf = ReplayBuffer(CAP, OBS, ACT, device="cuda")
        else:
            buf = PrioritizedReplayBuffer(CAP, OBS, ACT, device="cuda", max_batch=BATCH)
        fill(buf, CAP)
        eng = UpdateEngine(OBS, ACT, cfg)
        eng.reset_state()
        eng.attach_ring(buf)
        if kind == "per":
            eng.attach_per(buf)
        legs[kind] = (eng, buf)
    chunk = 1000
    rates = {"uniform": [], "per": []}
    for eng, _ in legs.values():
        eng.update(None, None, None, 50)
    torch.cuda.synchronize()
    for _ in range(args.repeats):
        for kind, (eng, _) in legs.items():
            us = event_time(lambda: eng.update(None, None, None, chunk), max(1, args.updates // chunk))
            rates[kind].append(chunk / (us * 1e-6))
    eng, _ = legs["per"]
    l0 = eng.launch_count()
    eng.update(None, None, None, 100)
    torch.cuda.synchronize()
    launches = (eng.launch_count() - l0) / 100.0

    tree = PrioritizedReplayBuffer(CAP, OBS, ACT, device="cuda", max_batch=65536)
    fill(tree, CAP)
    tree.slot_priorities()
    tree_us = {}
    gen = torch.Generator(device="cuda").manual_seed(1)
    for B in (256, 65536):
        idx = torch.empty(B, dtype=torch.int64, device="cuda")
        w = torch.empty(B, dtype=torch.float32, device="cuda")
        j = torch.randint(0, CAP, (B,), device="cuda", generator=gen)
        td = torch.rand(B, device="cuda", generator=gen) * 4
        ctr = [0]

        def sample():
            ctr[0] += 1
            E.check(tree._lib.sacx_per_sample(tree.per_handle, B, 0.4, None, 7, ctr[0], idx.data_ptr(), w.data_ptr()))

        def write_back():
            E.check(tree._lib.sacx_per_update_priorities(tree.per_handle, j.data_ptr(), td.data_ptr(), B))

        tree_us[str(B)] = {"sync_sample_us": round(event_time(sample, 200), 2), "write_back_us": round(event_time(write_back, 200), 2)}

    med = {k: statistics.median(v) for k, v in rates.items()}
    out = {
        "card": name, "power_limit": power,
        "workload": "bipedal shape: obs 24, act 4, 2x256, batch 256, 1M-slot ring; default kernel path " + legs["uniform"][0].path()[0],
        "updates_per_s": {k: {"median": round(med[k], 1), "min": round(min(v), 1), "max": round(max(v), 1), "repeats": len(v)}
                          for k, v in rates.items()},
        "per_update_overhead_us": round(1e6 / med["per"] - 1e6 / med["uniform"], 2),
        "tree_1M": tree_us,
        "launches_per_per_update": launches,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
