"""Per-phase timing of the fused update kernel (clock64 at barrier arrive / release for every CTA).
   python tools/phase_profile.py [workload] [steps]   -> prints a table; run on the GPU box."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the event trace of the row-parallel kernel is compiled into the debug library only
os.environ.setdefault("SACX_LIB", os.path.join(ROOT, "soft-actor-critic_b200", "lib", "libsacx_debug.so"))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-actor-critic_b200")]
import bench  # noqa: E402
import torch  # noqa: E402
from sac.agent import SAC  # noqa: E402
from sac import _engine as E  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else "bipedal"
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
w = dict(bench.WORKLOADS[wl])
w["fill"] = min(w["fill"], 200_000)
agent = SAC(bench.FakeEnv(w["obs"], w["act"]), bench.make_config(w, "device"))
agent.replay_buffer.push_batch(*bench.synth(w["fill"], w["obs"], w["act"]))
eng = agent.engine
eng.update(None, None, None, 50)
eng.sync()
gx, gy, smem = eng.grid()
cap = steps * 64 * gx * 10
buf = np.zeros(cap, dtype=np.uint64)
npz, ncta = C.c_int32(), C.c_int32()
eng._sync_stream()
E.check(eng.lib.sacx_debug_profile(eng.h, steps, buf.ctypes.data, cap, C.byref(npz), C.byref(ncta)))
P, G = npz.value, ncta.value
t = buf[: steps * P * G * 2].reshape(steps, P, G, 2).astype(np.int64)
arrive, release = t[..., 0], t[..., 1]
# per CTA: work(p) = arrive(p) - release(p-1); wait(p) = release(p) - arrive(p)
prev_release = np.concatenate([release[:, -1:, :][:, :, :] * 0, release[:, :-1, :]], axis=1)
skip = min(2, steps - 1)
work = (arrive - prev_release)[skip:, 1:, :]          # skip first steps and phase 0 (no previous release in-step)
wait = (release - arrive)[skip:, :, :]
span = (release[:, -2, :] - release[:, 0, :])[skip:]   # phases 1..P-2 span per step (same SM clock)
print(f"workload={wl} grid={gx} phases={P} clock~1.965GHz; cycles (median over steps)")
print("phase  work_max  work_med  work_min  wait_min  wait_med")
for p in range(P):
    wk = work[:, p - 1, :] if p >= 1 else None
    wt = wait[:, p, :]
    f = lambda a, fn: int(np.median(fn(a, axis=1))) if a is not None else -1
    print(f"{p:5d} {f(wk, np.max):9d} {f(wk, np.median):9d} {f(wk, np.min):9d} {f(wt, np.min):9d} {f(wt, np.median):9d}")
tot = np.median(release[2:, -2, 0] - release[1:-1, -2, 0]) if steps > 3 else 0
print("cycles per update (CTA0, release-to-release of phase P-2):", int(tot), "=", tot / 1.965e3, "us")

if len(sys.argv) > 3:
    for p in [int(x) for x in sys.argv[3].split(",")]:
        wk = np.median(work[:, p - 1, :], axis=0).astype(int)
        print(f"phase {p} work per CTA (cycles), CTA index = first tile index:")
        print(" ".join(f"{i}:{v}" for i, v in enumerate(wk)))

if eng.path()[0] == "rowpar":
    tr = buf[steps * P * G * 2:]
    n = int(tr[0])
    ev = tr[1: 1 + 2 * n].reshape(n, 2).astype(np.int64)
    print(f"event trace of CTA 0, last update ({n} events): tag  +cycles-since-previous  cycles-since-first")
    for i in range(n):
        print(f"  {ev[i, 0]:5d} {ev[i, 1] - ev[max(i - 1, 0), 1]:8d} {ev[i, 1] - ev[0, 1]:9d}")
    sys.exit(0)
t2 = buf[steps * P * G * 2: steps * P * G * 10].reshape(steps, P, G, 8).astype(np.int64)
print("intra-tile (CTA's last GEMM tile), median over steps and CTAs that ran a GEMM tile: load0  kloop  reduce  epilogue  total")
for p in range(P):
    x = t2[2:, p]
    ok = x[..., 4] > x[..., 0]
    if ok.sum() == 0:
        continue
    d = lambda a, b: int(np.median((x[..., a] - x[..., b])[ok]))
    print(f"{p:5d} {d(1,0):7d} {d(2,1):7d} {d(3,2):7d} {d(4,3):7d} {d(4,0):7d}")

