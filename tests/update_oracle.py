"""One fused SAC update of the engine, split into its pieces and compared with the float64 NumPy oracle (oracle/sac_numpy.py)
on the same float32 inputs. Shared by the -m gpu oracle tests of every update path (test_gpu_rowpar_oracle.py,
test_gpu_tiles_oracle.py); nothing here compares one CUDA path with another.

Why the comparisons are built the way they are:
- the fused plans never write `g.*` (Adam is fused into the dW tiles / the dW reduce). Every update starts from Adam moments
  m = 0, so the kernel stores m = fl(0.1f g) and g = m / 0.1f to one ulp: the gradients are read back from `m.*`, and `g.*`
  is NaN before the launch and must still be NaN after it (the gradient-only entry points must overwrite all of it);
- the critics' activations and deltas in the arena are overwritten by the critics' forward at (s, a~) before the launch ends,
  so the critics' gradients cannot be corrected row by row on the engine side. Their batch is drawn from ring rows that sit on
  no discontinuity instead (a relu / leaky_relu / selu pre-activation within 2e-5 max(1, rms) of zero in either critic at
  (s, a) or in the policy at s, or a raw log-std that close to a clamp bound). Device-RNG cases, whose batch the kernel draws,
  use tanh hidden layers and must meet no such row;
- kinks that exist only after the critic step (the critics at (s, a~), near-ties of Q1 and Q2) are flagged after the launch and
  subtracted from both actor gradients: from the engine's own `delta.pi.*`, `scr.dhead`, `batch.spi`, `act.pia.h*`, which
  nothing overwrites after the actor half, and from the oracle's;
- Adam's first steps amplify noise-level gradient elements to +-lr, so the update is pinned as arithmetic instead: float32
  `AdamState` on the recovered gradient must reproduce the new parameters and v to 2e-6.

`one_update(..., grads=True)` runs the gradient-only entry points instead (sample_batch, target, critic_step and actor_step
with grads_only, no apply in between): the same comparisons on the gradients the engine stores in `g.*`, without the optimiser,
Polyak and temperature checks.

`case(..., per={...})` runs prioritized replay (test_gpu_per_oracle.py): a PrioritizedReplayBuffer with loaded priorities is
attached and `update(None, eps1, eps2, 1)` lets the tree draw the batch. Every ring row on a discontinuity gets priority 0, which
the walk never takes; batch.idx must equal oracle/per_numpy.py's walk_f32 on the loaded leaves with per_uniform's stream, bit
for bit. The critic oracle weighs row k by float64 w = (p / p_min)^-beta(t) (dout, loss rows, q losses, gradients), the actor
and temperature stay unweighted, and duplicate rows are expected (sampling with replacement). The write-back, applied by the
next read of the priorities, must give each sampled slot (delta + eps)^alpha of its highest row at rel 2e-6 and leave every
other leaf's bits alone.

Bars (DESIGN.md section 2): rel-L2 2e-5 on per-row outputs, 5e-5 on gradients (with the bias bar of
test_gpu_baseline_configs._check_layer_grads), 2e-6 on the Adam arithmetic, 1e-6 absolute on log_alpha, bits on the gather
and on Polyak. Callers print the largest error per quantity (`report`), so the margin is visible.

Before every launch the per-update float scratch (`batch.*`, `out.*`, `scr.*`, `delta.*`, `act.*`, padding columns included)
is filled with NaN: an element the update reads without writing it shows up as a NaN or a mismatch.
"""
import numpy as np
import torch

from gpu_helpers import base_config, load_nets, read_net
from helpers import grads_without_rows, oracle_forward_backward, rel_l2
from test_gpu_parity import _random_nets

THR = 2e-5                                  # discontinuity distance, relative to max(1, rms) of the pre-activations
KINKED = ("relu", "leaky_relu", "selu")     # activations whose derivative jumps at z = 0
POISON = ("batch.", "out.", "scr.", "delta.", "act.")
# every switch that selects an update path or a variant of one: cleared before each case, then set from the case's env
SWITCHES = ("SACX_ROWPAR", "SACX_RP_TMA", "SACX_RP_DW_TMA", "SACX_RP_DW_VEC", "SACX_RP_GROUPS", "SACX_TC", "SACX_TC_MIN_BATCH",
            "SACX_TILE", "SACX_TC_HEADS", "SACX_TC_ROWS", "SACX_TC_POP")
F32 = np.float32
T = (0, 1, 39886)                           # Adam step counts before the update


# ----------------------------------------------------------------------------------------------------------------- cases
def case(obs, act, hp, hq, B, actfn="relu", out_act="identity", t=0, wrap=False, auto=True, lo=-20.0, hi=2.0, scale=1.0,
         ties=False, device_rng=False, env=None, per=None):
    """per: prioritized replay, a dict of alpha, beta (beta0), beta_steps, eps, profile ("spread" or "peaked") and optionally
    updates (start value of scal.updates: the draw counter and the beta schedule's t)."""
    return dict(obs=obs, act=act, hp=hp, hq=hq, B=B, actfn=actfn, out_act=out_act, t=t, wrap=wrap, auto=auto, lo=lo, hi=hi,
                scale=scale, ties=ties, device_rng=device_rng, env=dict(env or {}), per=dict(per) if per else None)


# ------------------------------------------------------------------------------------------------------------ helpers
def _np(t):
    return t.detach().cpu().numpy().copy()


def _mlp(sd, hidden, out):
    from oracle.sac_numpy import mlp_from_state_dict
    return mlp_from_state_dict(sd, hidden, out, np.float64)


def _near_zero(z):
    return (np.abs(z) < THR * max(1.0, float(np.sqrt(np.mean(z ** 2))))).any(axis=1)


def _kink_rows(mlp, cache):
    """Rows on a discontinuity of the backward: a hidden or output pre-activation near the derivative jump of relu /
    leaky_relu / selu."""
    amb = np.zeros(cache["z"][0].shape[0], bool)
    if mlp.hidden_act in KINKED:
        for z in cache["z"][:-1]:
            amb |= _near_zero(z)
    if mlp.out_act in KINKED:
        amb |= _near_zero(cache["z"][-1])
    return amb


def _clamp_rows(head, A, lo, hi):
    ls = head[:, A:]
    return ((np.abs(ls - lo) < THR * max(1.0, abs(lo))) | (np.abs(ls - hi) < THR * max(1.0, abs(hi)))).any(axis=1)


def _poison(eng):
    """NaN over every per-update float buffer, padding columns included (batch.idx too: its words become a huge index)."""
    for name, (off, rows, cols, ld, dtype) in eng.layout.items():
        if name.startswith(POISON):
            eng.arena[off: off + rows * ld * (1 if dtype == 0 else 2)].fill_(float("nan"))


def _bar(what, e, bar, worst):
    worst[what] = max(worst.get(what, 0.0), e)
    assert e < bar, f"{what}: {e:.3e} >= {bar:.1e}"


def _check_grads(what, eng_gW, eng_gb, ref_gW, ref_gb, g_deltas, g_inputs, o_deltas, o_inputs, flagged, worst):
    """Per-tensor gradients without the flagged rows (subtracted on both sides), bars of _check_layer_grads."""
    gW, gb = grads_without_rows(eng_gW, eng_gb, g_deltas, g_inputs, flagged)
    rW, rb = grads_without_rows(ref_gW, ref_gb, o_deltas, o_inputs, flagged)
    keep = ~flagged
    for l in range(len(rW)):
        _bar(f"{what}.W{l} grad", rel_l2(gW[l], rW[l]), 5e-5, worst)
        err = np.linalg.norm(gb[l] - rb[l])
        lim = 5e-5 * np.linalg.norm(rb[l]) + 5e-6 * np.linalg.norm(np.abs(o_deltas[l][keep]).sum(axis=0))
        worst[f"{what}.b grad (of bar)"] = max(worst.get(f"{what}.b grad (of bar)", 0.0), err / lim)
        assert err < lim, f"{what}.b{l} grad: |err| {err:.3e} >= {lim:.3e}"


def _engine_grads(eng, tag, n_lin, grads):
    """The gradient the engine computed: g.* after the gradient-only entry points, else m / 0.1f (m = 0 before the update)."""
    if grads:
        return read_net(eng, tag, n_lin, prefix="g.")
    m = read_net(eng, tag, n_lin, prefix="m.")
    return {k: v / F32(0.1) for k, v in m.items()}


def _check_adam(eng, tag, n_lin, before, v_before, step, lr, grads, worst):
    """float32 torch Adam (m = 0 before the step) on the recovered gradient reproduces the new parameters and v."""
    from oracle.sac_numpy import AdamState
    names = list(before.keys())
    params = [before[nm].copy() for nm in names]
    st = AdamState(lr, [np.zeros_like(p) for p in params], [v_before[nm].copy() for nm in names], step=step)
    st.apply(params, [grads[nm] for nm in names])
    got, got_v = read_net(eng, tag, n_lin), read_net(eng, tag, n_lin, prefix="v.")
    for i, nm in enumerate(names):
        _bar(f"{tag} adam param", rel_l2(got[nm], params[i]), 2e-6, worst)
        _bar(f"{tag} adam v", rel_l2(got_v[nm], st.v[i]), 2e-6, worst)


def report(label, c, flagged, worst):
    print(f"\n[{label}] obs {c['obs']} act {c['act']} pi {c['hp']} q {c['hq']} B {c['B']} {c['actfn']}/{c['out_act']} "
          f"env {c['env']}: flagged (ring rows at (s, a), actor batch rows) per update {flagged}")
    for q, e in sorted(worst.items()):
        print(f"    {q:34s} {e:.2e}")


# ------------------------------------------------------------------------------------------------------------- set-up
def setup(c, monkeypatch, seed):
    from sac.engine import UpdateEngine
    from sac.replay_buffer import ReplayBuffer
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in c["env"].items():
        monkeypatch.setenv(k, v)
    O, A, B = c["obs"], c["act"], c["B"]
    cap = max(3 * B, 200)
    cfg = base_config(hidden=c["hp"], q_hidden=c["hq"], act=c["actfn"], out_act=c["out_act"], auto=c["auto"], batch=B,
                      seed=seed, capacity=cap, alpha=0.13, log_std_min=c["lo"], log_std_max=c["hi"], action_scale=c["scale"])
    eng = UpdateEngine(O, A, cfg)
    rng = np.random.default_rng(seed)
    sds = _random_nets(O, A, c["hp"], c["hq"], seed=seed, scale=0.15)
    # moderate policy heads: at log-std << 0 the reference's float32 Gaussian term (z - mu)^2 / (2 sigma^2) cancels z - mu
    # down to a few bits (sigma eps below ulp(mu)), which a float64 oracle would measure instead of the kernel
    for nm in (f"net.{2 * len(c['hp'])}.weight", f"net.{2 * len(c['hp'])}.bias"):
        sds["pi"][nm] = sds["pi"][nm] * F32(0.25)
    if c["ties"]:
        sds["q2"] = {k: v.copy() for k, v in sds["q1"].items()}
    tgt = {}
    for tag in ("q1", "q2"):
        tgt[tag + "t"] = {k: (v * (1 + 0.05 * rng.standard_normal(v.shape))).astype(F32) for k, v in sds[tag].items()}
    if c["ties"]:
        tgt["q2t"] = {k: v.copy() for k, v in tgt["q1t"].items()}
    load_nets(eng, dict(sds, **tgt))
    eng.reset_state()
    eng.view("block.m").zero_()
    eng.view("block.v").copy_(torch.as_tensor(rng.uniform(1e-8, 1e-6, eng.view("block.v").shape).astype(F32)))
    if c["ties"]:
        for tag, n in (("q1", len(c["hq"]) + 1),):
            for l in range(n):
                for wb in "Wb":
                    eng.view(f"v.q2.{wb}{l}").copy_(eng.view(f"v.q1.{wb}{l}"))
    eng.view("scal.step").copy_(torch.full((4,), c["t"], dtype=torch.int64))
    eng.view("scal.log_alpha").fill_(float(np.log(0.13) + 0.3 * rng.standard_normal()))
    eng.view("scal.alpha_m").fill_(float(0.01 * rng.standard_normal()))
    eng.view("scal.alpha_v").fill_(float(rng.uniform(1e-3, 1e-1)))
    eng.refresh_alpha()
    # ring: a large share of episode ends; wrapped cases pushed past capacity (oldest slot != 0)
    n_push = cap + cap // 3 + 7 if c["wrap"] else cap - 5
    s = rng.standard_normal((n_push, O)).astype(F32)
    s2 = rng.standard_normal((n_push, O)).astype(F32)
    a = rng.uniform(-1, 1, (n_push, A)).astype(F32)
    r = rng.standard_normal(n_push).astype(F32)
    d = (rng.random(n_push) < 0.4).astype(F32)
    per = c.get("per")
    if per:
        from sac.replay_buffer import PrioritizedReplayBuffer
        rb = PrioritizedReplayBuffer(cap, O, A, alpha=per["alpha"], beta=per["beta"], beta_steps=per["beta_steps"], eps=per["eps"])
    else:
        rb = ReplayBuffer(cap, O, A)
    for lo in range(0, n_push, cap // 2):
        rb.push_batch(s[lo: lo + cap // 2], a[lo: lo + cap // 2], r[lo: lo + cap // 2], s2[lo: lo + cap // 2], d[lo: lo + cap // 2])
    eng.attach_ring(rb)
    if per:
        eng.attach_per(rb)
        eng.view("scal.updates").fill_(int(per.get("updates", 0)))
        n = min(n_push, cap)
        if per["profile"] == "peaked":                # a few slots hold most of the mass: many duplicate rows
            p = np.full(n, 1e-3)
            p[rng.choice(n, 6, replace=False)] = 10.0
        else:                                         # (delta + eps)^alpha, delta over four decades
            p = (10.0 ** rng.uniform(-3, 1, n) + per["eps"]) ** per["alpha"]
        leaves = np.zeros(cap, F32)
        leaves[per_slots(n_push, cap, n)] = p
        rb.load_slot_priorities(torch.as_tensor(leaves), float(leaves.max()))
    first = max(n_push - cap, 0)                      # logical position j of the ring = push number first + j
    ring = tuple(x[first:] for x in (s, a, r, s2, d))
    return eng, rb, ring, rng


def per_slots(pushes, cap, n):
    """Ring slot of logical positions 0 .. n-1."""
    from oracle import per_numpy as P
    return P.logical_to_slot(np.arange(n), pushes, cap)


def _state(eng, c):
    nq, npi = len(c["hq"]) + 1, len(c["hp"]) + 1
    st = {tag: read_net(eng, tag, n) for tag, n in (("pi", npi), ("q1", nq), ("q2", nq), ("q1t", nq), ("q2t", nq))}
    st["v"] = {tag: read_net(eng, tag, n, prefix="v.") for tag, n in (("pi", npi), ("q1", nq), ("q2", nq))}
    st["step"] = _np(eng.view("scal.step")).tolist()
    st["log_alpha"] = float(eng.view("scal.log_alpha").item())
    st["alpha_m"], st["alpha_v"] = float(eng.view("scal.alpha_m").item()), float(eng.view("scal.alpha_v").item())
    st["alpha_f32"] = float(eng.view("scal.alpha_f32").item())
    st["updates"] = int(eng.view("scal.updates").item())
    return st


def _pre_flags(st, c, ring):
    """Ring rows on a discontinuity of the critics' backward at (s, a) or of the policy's at s (pre-update state)."""
    s, a = ring[0].astype(np.float64), ring[1].astype(np.float64)
    x = np.concatenate([s, a], axis=1)
    flags = np.zeros(len(s), bool)
    for tag in ("q1", "q2"):
        q = _mlp(st[tag], c["actfn"], c["out_act"])
        flags |= _kink_rows(q, q.forward(x)[1])
    pi = _mlp(st["pi"], c["actfn"], c["out_act"])
    head, cache = pi.forward(s)
    return flags | _kink_rows(pi, cache) | _clamp_rows(head, c["act"], c["lo"], c["hi"])


# ---------------------------------------------------------------------------------------------------------------- one update
def one_update(eng, c, ring, rng, worst, grads=False):
    from oracle import device_rng
    from oracle.sac_numpy import squash_sample
    O, A, B = c["obs"], c["act"], c["B"]
    nq, npi = len(c["hq"]) + 1, len(c["hp"]) + 1
    st = _state(eng, c)
    pre = _pre_flags(st, c, ring)
    n_ring = len(ring[0])
    per = c.get("per")
    if per:
        # the tree draws the batch: every ring row on a discontinuity gets p = 0, which the walk never takes
        from oracle import per_numpy as P
        assert not grads and not c["device_rng"]
        buf = eng.per
        cap, pushes = buf.capacity, int(buf._lib.sacx_ring_pushes(buf.handle, 0))
        leaves, pmax = buf.slot_priorities()                 # applies the previous update's write-back
        leaves = leaves.cpu().numpy()
        leaves[per_slots(pushes, cap, n_ring)[pre]] = 0
        assert (leaves > 0).any()
        buf.load_slot_priorities(torch.as_tensor(leaves), pmax)
        e1 = rng.standard_normal((B, A)).astype(F32)
        e2 = rng.standard_normal((B, A)).astype(F32)
    elif c["device_rng"]:
        assert not grads
        idx = None
    else:
        good = np.flatnonzero(~pre)
        assert len(good) >= B
        idx = rng.choice(good, B, replace=False).astype(np.int64)
        e1 = rng.standard_normal((B, A)).astype(F32)
        e2 = rng.standard_normal((B, A)).astype(F32)
    _poison(eng)
    eng.view("block.g").fill_(float("nan"))          # fused: must stay NaN; gradient-only: every element must be written
    if grads:
        dev = lambda x: torch.as_tensor(x).cuda()
        eng.sample_batch(dev(idx))
        eng.target(dev(e1))
        eng.critic_step(None, grads_only=True)
        eng.actor_step(dev(e2), None, grads_only=True)
        eng.sync()
        m = eng.metrics()
        assert m["nonfinite"] == 0 and m["updates"] == st["updates"]
    elif c["device_rng"]:
        eng.update(None, None, None, 1)
        eng.sync()
        m = eng.metrics()
        idx = _np(eng.view("batch.idx")).ravel()
        seed = int(eng.view("scal.rng_seed").item())
        agent = int(eng.view("scal.rng_agent").view(torch.int32).item())
        want = device_rng.feistel_indices(B, n_ring, seed, st["updates"], agent)
        assert np.array_equal(idx, want), "device index stream != feistel_index"
        e1, e2 = _np(eng.view("batch.eps1")), _np(eng.view("batch.eps2"))
        for which, e in ((1, e1), (2, e2)):
            ref = np.array([[device_rng.philox_normal(seed, st["updates"], which, row, j, agent) for j in range(A)] for row in range(B)])
            ulps = np.abs(e - ref) / (np.spacing(F32(1)) * np.maximum(1.0, np.abs(ref)))
            worst["eps (float32 ulps of max(1,|x|))"] = max(worst.get("eps (float32 ulps of max(1,|x|))", 0.0), float(ulps.max()))
            assert ulps.max() <= 4, f"eps{which}: {ulps.max():.1f} ulps from philox_normal"
        assert not pre[idx].any(), f"device batch meets {int(pre[idx].sum())} rows on a discontinuity: pick another seed"
    elif per:
        dev = lambda x: torch.as_tensor(x).cuda()
        eng.update(None, dev(e1), dev(e2), 1)
        eng.sync()
        m = eng.metrics()
        idx = _np(eng.view("batch.idx")).ravel()
        seed = int(eng.view("scal.rng_seed").item())
        agent = int(eng.view("scal.rng_agent").view(torch.int32).item())
        slots = P.walk_f32(P.tree_f32(leaves), device_rng.per_uniforms(seed, st["updates"], B, agent))
        oldest = pushes % cap if pushes > cap else 0
        assert np.array_equal(idx, (slots - oldest) % cap), \
            f"{int((idx != (slots - oldest) % cap).sum())} of {B} sampled slots differ from walk_f32"
        assert (leaves[slots] > 0).all() and not pre[idx].any()
        p64 = leaves.astype(np.float64)
        beta = P.beta_at(st["updates"], float(F32(per["beta"])), per["beta_steps"])
        w = (p64[slots] / p64[p64 > 0].min()) ** -beta
        n_dup = B - len(np.unique(slots))
        print(f"    per: t {st['updates']} beta {beta:.6f} w in [{w.min():.3g}, {w.max():.3g}]; duplicate rows {n_dup}; "
              f"zero-priority (flagged) ring rows {int(pre.sum())}")
    else:
        m = eng.update_host(idx, e1, e2, 1)
    if not grads:
        assert m["nonfinite"] == 0 and m["updates"] == st["updates"] + 1
        assert torch.isnan(eng.view("block.g")).all(), "the fused update stored gradients in g.*"
    s, a, r, s2, d = (x[idx] for x in ring)

    # ---- gather: bits
    sa = _np(eng.view("batch.sa"))
    assert np.array_equal(sa, np.concatenate([s, a], axis=1)), "batch.sa"
    s2a = _np(eng.view("batch.s2a"))
    assert np.array_equal(s2a[:, :O], s2), "batch.s2a[:, :O]"
    assert np.array_equal(_np(eng.view("batch.r")).ravel(), r) and np.array_equal(_np(eng.view("batch.d")).ravel(), d)
    assert np.array_equal(_np(eng.view("batch.idx")).ravel(), idx)

    # ---- target, float64 on the pre-update state
    f64 = lambda x: np.asarray(x, np.float64)
    pi0 = _mlp(st["pi"], c["actfn"], c["out_act"])
    q1t, q2t = _mlp(st["q1t"], c["actfn"], c["out_act"]), _mlp(st["q2t"], c["actfn"], c["out_act"])
    alpha = st["alpha_f32"]
    head2, _ = pi0.forward(f64(s2))
    a2, lp2, _ = squash_sample(head2, f64(e1), c["lo"], c["hi"], c["scale"])
    x2 = np.concatenate([f64(s2), a2], axis=1)
    tq1, tq2 = q1t.forward(x2)[0][:, 0], q2t.forward(x2)[0][:, 0]
    y = f64(r) + 0.99 * (1 - f64(d)) * (np.minimum(tq1, tq2) - alpha * lp2)
    for name, got, ref in (("a'", s2a[:, O:], a2), ("logpi_next", eng.view("out.logpi_next"), lp2), ("tq1", eng.view("out.tq1"), tq1),
                           ("tq2", eng.view("out.tq2"), tq2), ("y", eng.view("out.y"), y)):
        _bar(name, rel_l2(got if isinstance(got, np.ndarray) else _np(got), ref), 2e-5, worst)

    # ---- critics
    # prioritized replay: loss (1/B) sum w diff^2 (w = (p / p_min)^-beta(t)); uniform: w = 1
    x = np.concatenate([f64(s), f64(a)], axis=1)
    wt = w if per else np.ones(B)
    for cc, tag in ((1, "q1"), (2, "q2")):
        q = _mlp(st[tag], c["actfn"], c["out_act"])
        qv, cache = q.forward(x)
        diff = qv[:, 0] - y
        _, cache, deltas, _ = oracle_forward_backward(q, x, (2 * wt * diff / B)[:, None])
        _bar("q", rel_l2(_np(eng.view(f"out.q{cc}")), qv[:, 0]), 2e-5, worst)
        _bar("dout", rel_l2(_np(eng.view(f"scr.dout{cc}"))[:, 0], deltas[-1][:, 0]), 2e-5, worst)
        _bar("q loss rows", rel_l2(_np(eng.view(f"scr.lossrow{cc}")), wt * diff * diff), 2e-5, worst)
        if not grads:
            ql = np.mean(wt * diff * diff)
            _bar("q loss", abs(m[f"q{cc}_loss"] - ql) / ql, 2e-5, worst)
        g = _engine_grads(eng, tag, nq, grads)
        ref = q.backward(cache, (2 * wt * diff / B)[:, None])
        no = np.zeros(B, bool)
        _check_grads(tag, [g[f"net.{2 * l}.weight"] for l in range(nq)], [g[f"net.{2 * l}.bias"] for l in range(nq)], ref[0], ref[1],
                     deltas, cache["h"][:nq], deltas, cache["h"][:nq], no, worst)
        if not grads:
            _check_adam(eng, tag, nq, st[tag], st["v"][tag], st["step"][cc], 3e-4, g, worst)

    # ---- Polyak: bits, from the engine's post-step critics
    if not grads:
        tau, omt = (F32(v) for v in _np(eng.view("scal.tau")).ravel())
        for tag in ("q1", "q2"):
            new, tnew = read_net(eng, tag, nq), read_net(eng, tag + "t", nq)
            for nm in new:
                assert np.array_equal(tnew[nm], tau * new[nm] + omt * st[tag + "t"][nm]), f"polyak {tag}t.{nm}"
    if c["ties"]:
        for nm, v in read_net(eng, "q1", nq).items():
            assert np.array_equal(v, read_net(eng, "q2", nq)[nm]), "tied critics diverged"

    # ---- actor: post-step critics (read exactly; unchanged by the gradient-only calls), pre-update policy and alpha
    post = {tag: _mlp(read_net(eng, tag, nq), c["actfn"], c["out_act"]) for tag in ("q1", "q2")}
    head, pcache = pi0.forward(f64(s))
    act_, lp, aux = squash_sample(head, f64(e2), c["lo"], c["hi"], c["scale"])
    xa = np.concatenate([f64(s), act_], axis=1)
    qa, ca, flags = [], [], _kink_rows(pi0, pcache) | _clamp_rows(head, A, c["lo"], c["hi"])
    for tag in ("q1", "q2"):
        v, cache = post[tag].forward(xa)
        qa.append(v[:, 0]); ca.append(cache)
        flags |= _kink_rows(post[tag], cache)
    dq = np.abs(qa[0] - qa[1])
    flags |= (dq > 0) & (dq < THR * max(1.0, float(np.sqrt(np.mean(qa[0] ** 2)))))
    w1 = np.where(qa[0] < qa[1], 1.0, np.where(qa[0] == qa[1], 0.5, 0.0))
    dx1 = post["q1"].backward(ca[0], (-w1 / B)[:, None], need_dx=True, need_dw=False)[2]
    dx2 = post["q2"].backward(ca[1], (-(1 - w1) / B)[:, None], need_dx=True, need_dw=False)[2]
    d_a = dx1[:, O:] + dx2[:, O:]
    tz, se, mask = aux["tz"], aux["se"], aux["mask"]
    dz = (alpha / B) * (2 * tz) + d_a * (c["scale"] * (1 - tz * tz))
    d_head = np.concatenate([dz, (se * dz - alpha / B) * mask], axis=1)
    _, pcache, pdeltas, _ = oracle_forward_backward(pi0, f64(s), d_head)
    keep = ~flags
    spi = _np(eng.view("batch.spi"))
    assert np.array_equal(spi[:, :O], s)
    _bar("a~", rel_l2(spi[:, O:], act_), 2e-5, worst)
    _bar("logpi", rel_l2(_np(eng.view("out.logpi")), lp), 2e-5, worst)
    q1_pi, q2_pi = _np(eng.view("out.q1_pi")).ravel(), _np(eng.view("out.q2_pi")).ravel()
    _bar("q_pi", max(rel_l2(q1_pi, qa[0]), rel_l2(q2_pi, qa[1])), 2e-5, worst)
    if c["ties"]:
        assert np.array_equal(q1_pi, q2_pi) and (qa[0] == qa[1]).all()
    dhead = _np(eng.view("scr.dhead"))
    _bar("dhead (unflagged rows)", rel_l2(dhead[keep], pdeltas[-1][keep]), 2e-5, worst)
    g_deltas = [_np(eng.view(f"delta.pi.{l}")) for l in range(npi - 1)] + [dhead]
    g_inputs = [spi[:, :O]] + [_np(eng.view(f"act.pia.h{l}")) for l in range(npi - 1)]
    for l in range(npi - 1):
        _bar("delta.pi (unflagged rows)", rel_l2(g_deltas[l][keep], pdeltas[l][keep]), 2e-5, worst)
    prow = alpha * lp - np.minimum(qa[0], qa[1])
    _bar("policy loss rows", rel_l2(_np(eng.view("scr.plossrow")), prow), 2e-5, worst)
    if not grads:
        # a mean of signed rows: relative to the mean of their magnitudes, which is what rounding of the rows adds up to
        _bar("policy loss (of mean |row|)", abs(m["policy_loss"] - prow.mean()) / np.abs(prow).mean(), 2e-5, worst)
    g = _engine_grads(eng, "pi", npi, grads)
    ref = pi0.backward(pcache, d_head)
    _check_grads("pi", [g[f"net.{2 * l}.weight"] for l in range(npi)], [g[f"net.{2 * l}.bias"] for l in range(npi)], ref[0], ref[1],
                 g_deltas, g_inputs, pdeltas, pcache["h"][:npi], flags, worst)
    if grads:
        return int(pre.sum()), int(flags.sum())
    _check_adam(eng, "pi", npi, st["pi"], st["v"]["pi"], st["step"][0], 3e-4, g, worst)
    if per:
        _check_write_back(eng, per, slots, leaves, pmax, worst)

    # ---- temperature
    la = float(eng.view("scal.log_alpha").item())
    if c["auto"]:
        lp_e = f64(_np(eng.view("out.logpi")).ravel())
        grad = -np.mean(lp_e - A)
        tt = st["step"][3] + 1
        am = st["alpha_m"] + 0.1 * (grad - st["alpha_m"])
        av = st["alpha_v"] * 0.999 + 0.001 * grad * grad
        la_ref = st["log_alpha"] - (3e-4 / (1 - 0.9 ** tt)) * (am / (np.sqrt(av) / np.sqrt(1 - 0.999 ** tt) + 1e-8))
        _bar("log_alpha (abs)", abs(la - la_ref), 1e-6, worst)
        _bar("alpha_m (abs)", abs(float(eng.view("scal.alpha_m").item()) - am), 1e-6, worst)
        _bar("alpha_v (rel)", abs(float(eng.view("scal.alpha_v").item()) - av) / av, 2e-6, worst)
    else:
        assert la == st["log_alpha"], "fixed temperature: log_alpha moved"
    return int(pre.sum()), int(flags.sum())


def _check_write_back(eng, per, slots, leaves, pmax, worst):
    """The update's deferred write-back, applied by the read: each sampled slot holds (delta + eps)^alpha of its highest row
    (delta in float64 from the engine's own out.q1 / q2 / y; rel 2e-6 for float32 powf), every other leaf keeps its bits,
    p_max is the float32 max."""
    from oracle import per_numpy as P
    q1, q2, y = (_np(eng.view(v)).ravel() for v in ("out.q1", "out.q2", "out.y"))
    pr = P.priority(P.td_delta(q1, q2, y), float(F32(per["alpha"])), float(F32(per["eps"])))
    after, pmax_after = eng.per.slot_priorities()
    after = after.cpu().numpy()
    last = {}
    for k, s in enumerate(slots.tolist()):
        last[s] = k                                   # the highest row wins a slot drawn more than once
    ss, ks = np.array(list(last)), np.array(list(last.values()))
    _bar("priority (rel)", float(np.max(np.abs(after[ss] - pr[ks]) / pr[ks])), 2e-6, worst)
    rest = np.ones(len(after), bool)
    rest[ss] = False
    assert np.array_equal(after[rest], leaves[rest]), "write-back changed a leaf it did not sample"
    assert pmax_after >= max(pmax, float(after.max()))
    _bar("p_max (rel)", abs(pmax_after - max(pmax, pr.max())) / max(pmax, pr.max()), 2e-6, worst)


def run_updates(eng, c, ring, rng, n=2, grads=False):
    """n updates, each from Adam m = 0 (v, the step counts and the rest carry over); returns (flagged rows, worst errors)."""
    worst, flagged = {}, []
    for k in range(n):
        if k:
            eng.view("block.m").zero_()
        flagged.append(one_update(eng, c, ring, rng, worst, grads=grads))
    return flagged, worst
