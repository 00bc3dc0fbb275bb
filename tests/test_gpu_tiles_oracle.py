"""-m gpu: the tile-parallel update (sacx_run_kernel, FFMA tiles 32x32 / 64x64, with the row ops of csrc/sacx_rowops.cuh) and the
tcgen05 tensor-core update (csrc/sacx_tc.cuh with the light row kernel sacx_rows_kernel) against the float64 NumPy oracle,
phase by phase, at the shapes and switches that select their code paths. Every shape the row-parallel kernel refuses runs here:
act > 8, obs > 123, batch > 512, widths other than 64/128/256, elu / gelu / selu hidden layers.

Same method and bars as test_gpu_rowpar_oracle.py (tests/update_oracle.py): one fused launch per update, two updates per case,
all per-update scratch NaN before each launch, the gather and Polyak in bits, gradients recovered from m = 0 as m / 0.1f with
`g.*` left untouched, the critics' batch off every discontinuity, the actor's kinked rows flagged after the launch.

Row-op variants. No API reports which variant a row op took, so the case table states it; the thresholds (staging area
`tsm_floats`: 18 688 floats in the 32x32 tile kernel, 34 816 in the 64x64 one, min(need, 12 288) in the light row kernel):
- tile_pi_head stages W_L when 2 A K + 2 A <= tsm (K = last policy hidden width): A = 32 at 32x32 -> K <= 291;
- OP_ACTOR_BWD stages when 2 A (H0 + K) <= tsm (H0 = first critic hidden width): 256/256 layers -> A <= 18 at 32x32;
- OP_Q_ROW stages when 4 K <= tsm (K = last critic hidden width): K <= 4 672 at 32x32;
- each staged op has a register-resident fast path (K <= 256, K % 4 == 0, 16-byte aligned rows) and a generic staged path;
  an unstaged op reads its weights from global memory.
Tensor-core fallbacks (`tc_skip`: FFMA or light-kernel ops inside tensor-core phases): layers wider than 256, dA with N < 16, a
policy head of width % 4 != 0 or SACX_TC_HEADS=0 (warp head op instead of head GEMM + OP_PI_TAIL), a critic head without the
epilogue projection (last critic width % 4 != 0 or SACX_TC_ROWS=0: OP_Q_ROW / OP_ACTOR_Q instead of OP_Q_TAIL + OP_DELTA),
first layers with K <= 32 (small_fwd_tile), dW with M <= 8 (small_dw_tile).
"""
import pytest

from gpu_helpers import base_config
from update_oracle import T, case, report, run_updates, setup

pytestmark = pytest.mark.gpu

NO_RP = {"SACX_ROWPAR": "0"}
D = ((256, 256), (256, 256))                 # the default workload's layers

# id: (case, tensor-core path expected, what it reaches)
CASES = {
    # ---- FFMA tiles, 32x32 (batch < 1024)
    "t32-default": (case(24, 4, *D, 256, t=T[0], env=NO_RP), False,
                    "fast row ops: head 2056, actor bwd 4096, q row 1024 floats staged; K = 256"),
    "t32-unaligned": (case(7, 5, (33, 17), (19, 23), 50, actfn="tanh", t=T[1], wrap=True), False,
                      "generic staged row ops: K = 17 / 23, nothing 16-byte aligned, ragged tiles"),
    "t32-humanoid": (case(376, 17, *D, 256, t=T[2], lo=-1.0, hi=0.3), False,
                     "A = 17 staged: head 8738, actor bwd 17408 <= 18688 (fast); active log-std clamp"),
    "t32-actor-bwd-unstaged": (case(40, 32, *D, 96, t=T[0], scale=2.5, lo=-1.0, hi=0.3), False,
                               "A = 32: actor bwd 32768 > 18688 unstaged; head 16448 staged fast; active clamp"),
    "t32-head-unstaged": (case(40, 32, (64, 320), (64, 64), 64, t=T[1], ties=True), False,
                          "A = 32, K = 320: head 20544 > 18688 unstaged (K > 256); exact Q1 = Q2 ties"),
    "t32-q-row-unstaged": (case(11, 3, (64, 64), (4800,), 64, t=T[2], wrap=True, auto=False), False,
                           "one 4800-wide critic layer: q row 19200 > 18688 unstaged, actor q 9600 staged generic; fixed alpha"),
    "t32-b513": (case(24, 4, *D, 513, t=T[1], wrap=True), False, "just past the row-parallel batch limit; last tile 1 row"),
    # ---- FFMA tiles, 64x64 (batch >= 1024, or SACX_TILE)
    "t32-b1023": (case(24, 4, *D, 1023, t=T[0]), False, "32x32 tiles one row below the switch"),
    "t64-b1024": (case(24, 4, *D, 1024, t=T[1], wrap=True), False, "64x64 tiles from 1024 rows"),
    "t32-forced-b1024": (case(17, 6, *D, 1024, t=T[2], env={"SACX_TILE": "small"}), False, "SACX_TILE=small at 1024"),
    "t64-forced-b256": (case(17, 6, *D, 256, t=T[0], scale=2.5, env=dict(NO_RP, SACX_TILE="large")), False,
                        "SACX_TILE=large at 256: staging area 34816"),
    # ---- saved pre-activations (tiles only)
    "z-elu": (case(24, 4, *D, 256, actfn="elu", out_act="tanh", t=T[1]), False, "elu hidden, tanh output"),
    "z-gelu": (case(17, 6, (128, 128), (128, 128), 300, actfn="gelu", out_act="elu", t=T[2], wrap=True), False,
               "gelu (erf) hidden, elu output"),
    "z-selu": (case(30, 3, (64, 64, 64), (64, 64, 64), 200, actfn="selu", out_act="selu", t=T[0], lo=-1.0, hi=0.3), False,
               "selu hidden and output (kinks flagged)"),
    # deepest plans the op table holds: the fused plan has 4 Lp + 12 Lq + 6 ops (MAX_OPS 112) in 2 Lp + 4 Lq + 4 phases
    # (MAX_PHASES 48); with at most 8 hidden layers per network the op count binds: (Lp, Lq) = (8, 6), (5, 7), (2, 8)
    "z-deepest-pi": (case(12, 2, (64,) * 8, (64,) * 6, 64, actfn="elu", t=T[1], wrap=True, auto=False), False,
                     "8 policy + 6 critic layers: 110 ops"),
    "z-deepest-q": (case(9, 3, (32, 32), (32,) * 8, 48, actfn="gelu", t=T[2]), False, "2 policy + 8 critic layers: 110 ops"),
    # ---- tensor core
    "tc-default": (case(24, 4, *D, 4096, t=T[0]), True,
                   "head GEMM + OP_PI_TAIL, critic projections + OP_Q_TAIL + OP_DELTA, small_fwd (K0 = 28), small_dw (M = 1, 8)"),
    "tc-b129": (case(24, 4, *D, 129, t=T[1], wrap=True, lo=-1.0, hi=0.3, env={"SACX_TC_MIN_BATCH": "128"}), True,
                "second 128-row tile holds one row; active clamp"),
    "tc-a32-warp-rows": (case(40, 32, *D, 256, t=T[2], scale=2.5, lo=-1.0, hi=0.3,
                              env={"SACX_TC_MIN_BATCH": "256", "SACX_TC_HEADS": "0", "SACX_TC_ROWS": "0"}), True,
                         "light kernel (12288): warp head 16448 and actor bwd 32768 unstaged, q row staged; active clamp"),
    "tc-mixed": (case(20, 3, (512, 12, 250), (64, 254), 1024, t=T[1], env={"SACX_TC_MIN_BATCH": "1024"}), True,
                 "512-wide layer FFMA, dA N = 12 FFMA, policy head K = 250 (warp head), critic K = 254 (no projection)"),
    "tc-obs216": (case(216, 4, *D, 2048, t=T[2], wrap=True, env={"SACX_TC_MIN_BATCH": "2048"}), True,
                  "first layers K = 216 / 220 on tensor cores"),
    "tc-tanh": (case(24, 4, *D, 1024, actfn="tanh", t=T[0], ties=True, auto=False, env={"SACX_TC_MIN_BATCH": "1024"}), True,
                "tanh hidden; exact ties; fixed alpha"),
    "tc-leaky": (case(24, 4, (128, 256), (256, 128), 1024, actfn="leaky_relu", t=T[1], wrap=True,
                      env={"SACX_TC_MIN_BATCH": "1024"}), True, "leaky_relu hidden"),
    "tc-elu-refused": (case(24, 4, *D, 256, actfn="elu", out_act="tanh", t=T[2], env={"SACX_TC": "1", "SACX_TC_MIN_BATCH": "256"}),
                       False, "SACX_TC=1 with elu: tiles"),
    # ---- device RNG (tanh: no kinks the kernel's own batch could meet)
    "devrng-tiles": (case(17, 3, (48, 40), (40, 48), 70, actfn="tanh", t=T[1], wrap=True, device_rng=True), False,
                     "OP_PI_HEAD normals"),
    "devrng-tc": (case(24, 4, (128, 128), (128, 128), 256, actfn="tanh", t=T[2], device_rng=True,
                       env={"SACX_TC_MIN_BATCH": "128"}), True, "OP_PI_TAIL normals"),
}


def _check_path(eng, tc, updated):
    kind, why = eng.path()
    assert kind == "tiles", (kind, why)
    on, tc_why, launches = eng.tensor_core()
    assert on == tc, tc_why
    assert (launches > 0) == (tc and updated), launches


@pytest.mark.parametrize("name", list(CASES))
def test_tiles_update_vs_float64_oracle(name, monkeypatch):
    c, tc, what = CASES[name]
    seed = 2000 + 17 * c["obs"] + c["act"]
    eng, rb, ring, rng = setup(c, monkeypatch, seed)
    _check_path(eng, tc, False)
    flagged, worst = run_updates(eng, c, ring, rng)
    _check_path(eng, tc, True)
    report(f"{name}: {'tensor core' if tc else 'tiles'}: {what}", c, flagged, worst)


def test_tc_refuses_saved_preactivations(monkeypatch):
    """elu forced onto the tensor-core path: the engine runs the FFMA tiles and says why."""
    c = CASES["tc-elu-refused"][0]
    eng, _, _, _ = setup(c, monkeypatch, 1)
    assert eng.path() == ("tiles", "hidden activation needs saved pre-activations")
    assert eng.tensor_core() == (False, "hidden activation needs saved pre-activations", 0)


# ------------------------------------------------------------------------------------ gradient-only entry points, split batch
@pytest.mark.parametrize("B", [2049, 2560])
@pytest.mark.parametrize("tc", [False, True], ids=["tiles", "tc"])
def test_gradient_entry_points_vs_float64_oracle(B, tc, monkeypatch):
    """sample_batch, target, critic_step(grads_only) and actor_step(grads_only): g.* against float64. From 2048 rows the
    gradient-only dW ops split the batch into 512-row chunks accumulated with atomics (DW_ATOMIC): at 2049 the last chunk holds
    one row."""
    c = case(24, 4, *D, B, t=T[1], wrap=B == 2560, env={"SACX_TC_MIN_BATCH": "2048"} if tc else {"SACX_TC": "0"})
    eng, rb, ring, rng = setup(c, monkeypatch, 3000 + B)
    assert eng.path()[0] == "tiles" and eng.tensor_core()[0] == tc
    flagged, worst = run_updates(eng, c, ring, rng, grads=True)
    assert (eng.tensor_core()[2] > 0) == tc
    report(f"grads only, {'tensor core' if tc else 'tiles'}", c, flagged, worst)


# --------------------------------------------------------------------------------------------------------- op-table limit
@pytest.mark.parametrize("hp,hq,ok", [
    ((64,) * 8, (64,) * 6, True), ((64,) * 8, (64,) * 7, False),
    ((64,) * 5, (64,) * 7, True), ((64,) * 6, (64,) * 7, False),
    ((64,) * 2, (64,) * 8, True), ((64,) * 3, (64,) * 8, False),
])
def test_op_table_depth_limit(hp, hq, ok, monkeypatch):
    """The deepest networks the fused plan's op table holds are accepted; one layer more is refused with the op-table message."""
    from sac.engine import UpdateEngine
    for k in ("SACX_ROWPAR", "SACX_TC", "SACX_TC_MIN_BATCH"):
        monkeypatch.delenv(k, raising=False)
    cfg = base_config(hidden=hp, q_hidden=hq, batch=64)
    if ok:
        assert UpdateEngine(12, 2, cfg).path()[0] == "tiles"
    else:
        with pytest.raises(ValueError, match=r"network too deep for the op table \(MAX_OPS/MAX_PHASES\)"):
            UpdateEngine(12, 2, cfg)
