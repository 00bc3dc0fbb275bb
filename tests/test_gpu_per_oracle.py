"""-m gpu: prioritized replay (csrc/sacx_per.cuh and the weighted critic rows of the three update kernels) against the float32
restatement and the float64 oracle of oracle/per_numpy.py.

Sampler. The walk uses adds, one correctly rounded divide and one multiply (the library is built without fast-math), so the
slot of every draw equals `walk_f32` on the same float32 leaves, bit for bit, and no draw takes a slot with p = 0. The weight
w = powf(p / p_min, -beta) is compared with float64 (p / p_min)^-beta at rel 2e-6:
- the float32 divide: 2^-24 relative on the ratio, beta 2^-24 <= 6e-8 on w;
- powf: at most 4 ulp (CUDA C Programming Guide, single-precision functions): 4 2^-23 = 4.8e-7;
- beta as a float32: |d beta| <= 2^-24 beta, times |ln(p / p_min)| <= ln(1e4): 5.5e-7 at beta = 1.
That sums to 1.1e-6; each case prints its largest weight error.

Weighted update. tests/update_oracle.py with `per`: the tree draws the batch (zero priority on every ring row on a
discontinuity), batch.idx must equal walk_f32 on the loaded leaves with per_uniform's stream, the critic oracle weighs its rows
by float64 (p / p_min)^-beta(t), and the write-back that the next read applies must hold (delta + eps)^alpha of the update's
own q1 / q2 / y. Each case names the site of the weight it reaches:
- rp_target_critic<true> (csrc/sacx_rowpar.cuh): the weight of global row c.row0 + mm, in every round and grouping of row
  blocks;
- tile_q_row (csrc/sacx_rowops.cuh): w_in, loaded with the row's scalars, in its staged-fast, staged-generic and unstaged
  variants (the thresholds are in test_gpu_tiles_oracle.py);
- tile_q_tail (OP_Q_TAIL + OP_DELTA on the tensor-core path), and the light kernel's tile_q_row with SACX_TC_ROWS=0.

Chain. Five single updates with pushes between them and no read of the tree, so each update's write-back lands in the next
update's tree launch together with the new pushes and the incremental propagation. A float64 oracle carries the leaves; the
device's float32 leaves differ from it by the float32 priorities (rel 2e-6), so a draw within
(2e-6 + (3 + 17 depth) 2^-24) total of a prefix boundary (test_per_oracle_cpu.py) may take either neighbour and is counted.
"""
import numpy as np
import pytest
import torch

from update_oracle import T, case, report, run_updates, setup

pytestmark = pytest.mark.gpu
F32 = np.float32
U24 = 2.0 ** -24


# ------------------------------------------------------------------------------------------------------------ sampler
def _buf(cap, **kw):
    from sac.replay_buffer import PrioritizedReplayBuffer
    return PrioritizedReplayBuffer(cap, 3, 2, device="cuda", **kw)


def _push(buf, n, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    for i in range(0, n, buf.capacity):
        k = min(n - i, buf.capacity)
        r = lambda *s: torch.randn(*s, device="cuda", generator=g)
        buf.push_device(r(k, 3), r(k, 2), r(k), r(k, 3), (r(k) > 0).float())
    buf.slot_priorities()


def _profile(rng, n, zeros=0.1):
    """(delta + eps)^0.6 with delta over four decades, zeros mixed in."""
    p = ((10.0 ** rng.uniform(-3, 1, n) + 1e-6) ** 0.6).astype(F32)
    p[rng.random(n) < zeros] = 0
    p[rng.integers(0, n)] = F32(2.0)
    return p


def _pushes(buf):
    return int(buf._lib.sacx_ring_pushes(buf.handle, 0))


def _check_sample(buf, leaves, idx, w, U, beta, worst):
    from oracle import per_numpy as P
    slots = P.logical_to_slot(idx, _pushes(buf), buf.capacity)
    want = P.walk_f32(P.tree_f32(leaves), U)
    assert np.array_equal(slots, want), f"{int((slots != want).sum())} of {len(U)} slots differ from walk_f32"
    assert (leaves[slots] > 0).all(), "a draw took an empty slot"
    p = leaves.astype(np.float64)
    ref = (p[slots] / p[p > 0].min()) ** -float(beta)
    e = float(np.max(np.abs(w - ref) / ref))
    worst["w"] = max(worst.get("w", 0.0), e)
    assert e < 2e-6, f"weights: {e:.2e}"


SAMPLER = [  # (capacity, pushes, batches)
    (1, 1, (1, 7)),
    (31, 20, (1, 7, 256)),                    # depth 1, partly filled
    (32, 32, (7, 256, 4096)),                 # one full level
    (33, 33 + 20, (7, 256)),                  # one leaf past a level, wrapped
    (1025, 1025, (256, 4096)),
    (1025, 700, (7, 256)),
    (5000, 7300, (1, 256, 4096)),             # wrapped, not a multiple of 32
    (1 << 20, 1 << 20, (256, 65536)),         # 65 536 rows: more than the capped grid's warps, each walks several rows
]


@pytest.mark.parametrize("cap,pushes,batches", SAMPLER, ids=[f"cap{c}-pushes{p}" for c, p, _ in SAMPLER])
def test_sampler_matches_walk_f32(cap, pushes, batches):
    from oracle import device_rng as R
    from sac import _engine as E
    rng = np.random.default_rng(cap + pushes)
    buf = _buf(cap)
    _push(buf, pushes)
    n = min(pushes, cap)
    oldest = pushes % cap if pushes > cap else 0
    leaves = np.zeros(cap, F32)
    leaves[(oldest + np.arange(n)) % cap] = _profile(rng, n)
    buf.load_slot_priorities(torch.as_tensor(leaves), float(leaves.max()))
    worst, draws = {}, 0
    for B in batches:
        for beta in (0.4, 1.0):
            U = rng.random(B).astype(F32)
            U[0], U[-1] = 0.0, F32(1 - U24)                      # edge draws: u = 0 and u -> total
            idx, w = buf.sample_with_uniforms(torch.as_tensor(U), beta)
            _check_sample(buf, leaves, idx.cpu().numpy(), w.cpu().numpy(), U, F32(beta), worst)
            draws += B
        # the Philox form: per_uniform(seed, counter, k, agent 0)
        idx = torch.empty(B, dtype=torch.int64, device="cuda")
        w = torch.empty(B, dtype=torch.float32, device="cuda")
        E.check(buf._lib.sacx_per_sample(buf.per_handle, B, 0.7, None, 99, 12345 + B, idx.data_ptr(), w.data_ptr()))
        _check_sample(buf, leaves, idx.cpu().numpy(), w.cpu().numpy(), R.per_uniforms(99, 12345 + B, B, 0), F32(0.7), worst)
        draws += B
    print(f"\n[sampler cap {cap} pushes {pushes}] {draws} draws, slots equal walk_f32; largest weight error {worst['w']:.2e} "
          f"(bar 2e-6)")


def test_rounding_never_takes_an_empty_slot():
    """The two float32 traps of test_per_oracle_cpu.py on the device: a draw that rounding puts at the start of a child whose
    first slot is empty, and a last-stratum draw past the scanned sum of a partly filled ring. Before the walk required
    p > 0 of the child it takes, both drew an empty slot (weight inf)."""
    from test_per_oracle_cpu import end_trap, start_trap
    for leaves, U, want in (start_trap() + (33,), end_trap() + (19,)):
        buf = _buf(len(leaves))
        _push(buf, len(leaves))
        buf.load_slot_priorities(torch.as_tensor(leaves), float(leaves.max()))
        idx, w = buf.sample_with_uniforms(torch.as_tensor(U), 1.0)
        assert int(idx[0]) == want and np.isfinite(float(w[0])), (int(idx[0]), float(w[0]))


# ----------------------------------------------------------------------------------------------- weighted update per path
FIXED = dict(alpha=0.6, beta=0.4, beta_steps=0, eps=1e-6, profile="spread")           # beta0 = 0.4 held
ONE = dict(FIXED, beta=1.0)                                                           # beta = 1
BELOW = dict(FIXED, beta_steps=1000, updates=998)                                     # t = 998, 999: just below
ACROSS = dict(FIXED, beta_steps=1000, updates=999)                                    # t = 999, then 1000: beta -> 1
PEAKED = dict(FIXED, alpha=0.7, profile="peaked")                                    # six slots hold most of the mass
D = ((256, 256), (256, 256))
NO_RP = {"SACX_ROWPAR": "0"}

# id: (case, path, site)
CASES = {
    "rp-default": (case(24, 4, *D, 256, t=T[0], per=FIXED), "rowpar", "rp_target_critic<true>, one round of row blocks"),
    "rp-b1": (case(1, 1, (64, 64), (64, 64), 1, actfn="identity", t=T[1], wrap=True, per=ONE), "rowpar",
              "rp_target_critic<true>, one row"),
    "rp-row5": (case(62, 3, *D, 289, t=T[1], scale=2.5, per=BELOW), "rowpar",
                "rp_target_critic<true>, B 289: two rounds of row groups, 32x32 dW"),
    "rp-row8": (case(123, 8, (128, 128), (256, 64), 512, t=T[2], wrap=True, auto=False, per=ACROSS), "rowpar",
                "rp_target_critic<true>, A 8, cp.async; beta crosses 1"),
    "rp-row3-tanh": (case(30, 3, (128, 64), (64, 128), 17, out_act="tanh", t=T[2], per=ONE), "rowpar",
                     "rp_target_critic<true> with a tanh output: act' times w"),
    "rp-groups1": (case(24, 4, *D, 256, t=T[1], per=BELOW, env={"SACX_RP_GROUPS": "1"}), "rowpar",
                   "rp_target_critic<true>, SACX_RP_GROUPS=1"),
    "rp-groups5": (case(24, 4, *D, 256, t=T[2], wrap=True, per=ONE, env={"SACX_RP_GROUPS": "5"}), "rowpar",
                   "rp_target_critic<true>, SACX_RP_GROUPS=5"),
    "rp-no-tma": (case(24, 4, *D, 256, t=T[0], per=ACROSS, env={"SACX_RP_TMA": "0"}), "rowpar",
                  "rp_target_critic<true>, SACX_RP_TMA=0"),
    "rp-peaked": (case(24, 4, *D, 256, t=T[1], wrap=True, per=PEAKED), "rowpar",
                  "rp_target_critic<true>; many duplicate rows: highest row wins the write-back"),
    "t32-default": (case(24, 4, *D, 256, t=T[0], per=ONE, env=NO_RP), "tiles", "tile_q_row staged fast (K 256)"),
    "t32-unaligned": (case(7, 5, (33, 17), (19, 23), 50, actfn="tanh", t=T[1], wrap=True, per=ACROSS), "tiles",
                      "tile_q_row staged generic (K 23)"),
    "t32-q-row-unstaged": (case(11, 3, (64, 64), (4800,), 64, t=T[2], wrap=True, auto=False, per=FIXED), "tiles",
                           "tile_q_row unstaged (K 4800)"),
    "t64-b1024": (case(24, 4, *D, 1024, t=T[1], wrap=True, per=BELOW), "tiles", "tile_q_row in the 64x64 tile kernel"),
    "tc-default": (case(24, 4, *D, 4096, t=T[0], per=ONE), "tc", "tile_q_tail + OP_DELTA"),
    "tc-b129": (case(24, 4, *D, 129, t=T[1], wrap=True, lo=-1.0, hi=0.3, per=ACROSS, env={"SACX_TC_MIN_BATCH": "128"}), "tc",
                "tile_q_tail, second 128-row tile holds one row"),
    "tc-q-row": (case(24, 4, *D, 256, t=T[2], per=FIXED, env={"SACX_TC_MIN_BATCH": "256", "SACX_TC_ROWS": "0"}), "tc",
                 "light kernel tile_q_row (SACX_TC_ROWS=0)"),
}


@pytest.mark.parametrize("name", list(CASES))
def test_weighted_update_vs_float64_oracle(name, monkeypatch):
    c, path, site = CASES[name]
    eng, rb, ring, rng = setup(c, monkeypatch, 4000 + 17 * c["obs"] + c["act"])
    kind, why = eng.path()
    assert kind == ("rowpar" if path == "rowpar" else "tiles"), (kind, why)
    assert eng.tensor_core()[0] == (path == "tc")
    flagged, worst = run_updates(eng, c, ring, rng)
    report(f"{name}: {path}: {site}", c, flagged, worst)


# ------------------------------------------------------------------------------------------- chain through the write-back
CHAIN = {
    "rowpar": (case(24, 4, *D, 256, actfn="tanh", t=T[1], per=dict(FIXED, beta_steps=3, updates=1)), {}),
    "tc": (case(24, 4, *D, 256, actfn="tanh", t=T[1], wrap=True, per=dict(FIXED, beta_steps=3, updates=1)),
           {"SACX_TC_MIN_BATCH": "256"}),
}


@pytest.mark.parametrize("name", list(CHAIN))
def test_chain_through_the_deferred_write_back(name, monkeypatch):
    """update, no pushes, update, 37 pushes, update, half a ring (overwrites slots the last update sampled while their
    write-back is pending), update, a ring and 50 more (the reset), update; beta = 0.4 + 0.6 t / 3 for t = 1 .. 5."""
    from oracle import device_rng as R
    from oracle import per_numpy as P
    c, env = CHAIN[name]
    c = dict(c, env=env)
    per = c["per"]
    eng, rb, ring, rng = setup(c, monkeypatch, 5000 + len(name))
    assert eng.tensor_core()[0] == (name == "tc") and eng.path()[0] == ("rowpar" if name == "rowpar" else "tiles")
    O, A, B, cap = c["obs"], c["act"], c["B"], rb.capacity
    alpha, eps = float(F32(per["alpha"])), float(F32(per["eps"]))
    L, pmax = rb.slot_priorities()
    L, pmax = L.cpu().numpy().astype(np.float64), float(pmax)
    seen = _pushes(rb)
    depth = len(P.tree_f32(np.zeros(cap, F32))) - 1
    seed = int(eng.view("scal.rng_seed").item())
    agent = int(eng.view("scal.rng_agent").view(torch.int32).item())
    pending, flagged, worst = None, [], {}
    for step, n_push in enumerate((0, 37, cap // 2, cap + 50, None)):
        pushes = _pushes(rb)
        if pending is not None:                            # what this update's tree launch applies before it samples
            slots, pr = pending
            pmax = max(pmax, float(pr.max()))
            n_new = pushes - seen
            if n_new >= cap:
                L[:] = 0
                L[:min(pushes, cap)] = pmax
            else:
                new = (seen + np.arange(n_new)) % cap
                is_new = np.zeros(cap, bool); is_new[new] = True
                for k, s in enumerate(slots):
                    if not is_new[s]:
                        L[s] = pr[k]                         # rows in order: the highest row wins
                L[new] = pmax
        seen = pushes
        t = int(eng.view("scal.updates").item())
        e1 = torch.as_tensor(rng.standard_normal((B, A)).astype(F32)).cuda()
        e2 = torch.as_tensor(rng.standard_normal((B, A)).astype(F32)).cuda()
        eng.update(None, e1, e2, 1)
        eng.sync()
        assert eng.metrics()["nonfinite"] == 0
        idx = eng.view("batch.idx").cpu().numpy().ravel()
        slots = P.logical_to_slot(idx, pushes, cap)
        u = P.strata_u(R.per_uniforms(seed, t, B, agent), L.sum())
        tol = (2e-6 + (3 + 17 * depth) * U24) * L.sum()
        near = P.boundary_rows(L, u, tol)
        want = P.sample(L, u)
        assert np.array_equal(slots[~near], want[~near]), f"update {step}: {int((slots != want)[~near].sum())} draws differ"
        assert ((slots >= P.sample(L, np.maximum(u - tol, 0))) & (slots <= P.sample(L, u + tol))).all()
        assert (L[slots] > 0).all()
        flagged.append(int(near.sum()))
        # the weights the critic loss used: lossrow / diff^2 (one float32 rounding) against (p / p_min)^-beta(t)
        q1, y, lr = (eng.view(v).cpu().numpy().ravel() for v in ("out.q1", "out.y", "scr.lossrow1"))
        d2 = (q1 - y) * (q1 - y)
        ok = d2 > 0
        beta = P.beta_at(t, float(F32(per["beta"])), per["beta_steps"])
        w = (L[slots] / L[L > 0].min()) ** -beta
        e = float(np.max(np.abs(lr[ok] / d2[ok].astype(np.float64) - w[ok]) / w[ok]))
        worst["w (lossrow / diff^2)"] = max(worst.get("w (lossrow / diff^2)", 0.0), e)
        assert e < 1e-5, f"update {step} (t {t}, beta {beta}): weights {e:.2e} from the schedule"
        q2 = eng.view("out.q2").cpu().numpy().ravel()
        pending = (slots, P.priority(P.td_delta(q1, q2, y), alpha, eps))
        if n_push:
            s = rng.standard_normal((n_push, O)).astype(F32)
            a = rng.uniform(-1, 1, (n_push, A)).astype(F32)
            for lo in range(0, n_push, cap // 2):
                k = slice(lo, lo + cap // 2)
                rb.push_batch(s[k], a[k], np.ones(len(s[k]), F32), s[k], np.zeros(len(s[k]), F32))
    # the last write-back, applied by the read
    slots, pr = pending
    for k, s in enumerate(slots):
        L[s] = pr[k]
    pmax = max(pmax, float(pr.max()))
    got, gmax = rb.slot_priorities()
    got = got.cpu().numpy()
    assert np.array_equal(got == 0, L == 0)
    e = float(np.max(np.abs(got[L > 0] - L[L > 0]) / L[L > 0]))
    worst["leaves (rel)"] = e
    worst["p_max (rel)"] = abs(gmax - pmax) / pmax
    assert e < 2e-6 and worst["p_max (rel)"] < 2e-6
    print(f"\n[chain {name}] draws within the boundary bound per update: {flagged}")
    for q, v in sorted(worst.items()):
        print(f"    {q:34s} {v:.2e}")
