"""-m gpu: the row-parallel update (csrc/sacx_rowpar.cuh) against the float64 NumPy oracle, phase by phase, across the shapes
and options that select its code paths.

One fused launch (`update_host(idx, eps1, eps2, 1)`, or device RNG) is split into its pieces and every piece is compared with
oracle/sac_numpy.py in float64 on the same float32 inputs (tests/update_oracle.py: how and why, the bars); nothing here compares
one CUDA path with another.
"""
import pytest

from gpu_helpers import base_config
from update_oracle import T, case, report, run_updates, setup

pytestmark = pytest.mark.gpu

ROWS = {
    1: case(24, 4, (256, 256), (256, 256), 256, t=T[0]),                                   # default workload, vector dW tile
    2: case(1, 1, (64, 64), (64, 64), 1, actfn="identity", t=T[1], wrap=True),            # one row, K = 1 dW, smallest record
    3: case(30, 3, (128, 64), (64, 128), 17, out_act="tanh", t=T[2]),                      # gather W = 65; 2nd row block: 1 row
    4: case(61, 4, (128, 128), (256, 256), 288, t=T[0], wrap=True, lo=-1.0, hi=0.3),       # W = 128, reload ldx 76; 18 blocks
    5: case(62, 3, (256, 256), (256, 256), 289, t=T[1], scale=2.5),                        # gather W = 129; two rounds; 32x32 dW
    # rows 6-8: with 256-wide critics AND a 256-wide policy the shared memory runs out above obs 100 (see the boundary test);
    # a 64-wide second critic layer keeps the 256-wide first layer (TMA-eligible slices) inside the budget up to obs 123
    6: case(116, 4, (64, 128), (256, 64), 100, out_act="elu", t=T[2], wrap=True),         # ldx 124; critic K0 = 120
    7: case(120, 4, (128, 128), (256, 64), 64, t=T[0]),                                    # K0 = 124; reload ldx 132
    8: case(123, 8, (128, 128), (256, 64), 512, t=T[1], wrap=True),                       # W = 256, K0 = 131 cp.async; A = 8
    9: case(117, 4, (256, 64), (64, 256), 48, out_act="selu", t=T[2]),                     # reload ldx 132 with 64-wide layers
    10: case(20, 7, (64, 64, 64), (64, 64, 64), 33, actfn="tanh", t=T[0], wrap=True),      # act 7, three layers, tanh
    11: case(9, 5, (256, 64, 128), (64, 128, 256), 40, actfn="leaky_relu", t=T[1], ties=True),  # head class 16, lower edge
    12: case(12, 2, (64,) * 4, (64,) * 4, 64, t=T[2], wrap=True, auto=False),              # deepest: 2 Lq + Lp = 12
    14: case(24, 4, (256, 256), (256, 256), 1024, t=T[1], wrap=True, env={"SACX_ROWPAR": "1"}),   # FFMA dW, 64 blocks
}
FALLBACKS = [{"SACX_RP_TMA": "0"}, {"SACX_RP_DW_TMA": "0"}, {"SACX_RP_DW_VEC": "0"}, {"SACX_RP_GROUPS": "1"},
             {"SACX_RP_GROUPS": "5"}]
DEVICE_RNG = {
    "a1": case(3, 1, (64, 64), (64, 64), 37, actfn="tanh", t=T[1], wrap=True, device_rng=True),
    "a7": case(20, 7, (64, 64, 64), (64, 64, 64), 33, actfn="tanh", t=T[2], device_rng=True),
    "a8": case(17, 8, (128, 128), (128, 128), 50, actfn="tanh", t=T[0], wrap=True, device_rng=True),
}

PARAMS = [pytest.param(ROWS[k], id=f"row{k}") for k in ROWS]
PARAMS += [pytest.param(dict(ROWS[k], env=dict(ROWS[k]["env"], **fb)), id=f"row{k}-" + "-".join(f"{a}={b}" for a, b in fb.items()))
           for k in (1, 5, 8, 12) for fb in FALLBACKS]
PARAMS += [pytest.param(c, id=f"devrng-{k}") for k, c in DEVICE_RNG.items()]


@pytest.mark.parametrize("c", PARAMS)
def test_rowpar_update_vs_float64_oracle(c, monkeypatch):
    seed = 1000 + 17 * c["obs"] + c["act"]
    eng, rb, ring, rng = setup(c, monkeypatch, seed)
    kind, why = eng.path()
    assert kind == "rowpar", (kind, why)
    report(kind, c, *run_updates(eng, c, ring, rng))


# ------------------------------------------------------------------------------------------------------ eligibility edges
@pytest.mark.parametrize("obs,act,hp,hq,B,kind,why", [
    (123, 8, (128, 128), (256, 64), 64, "rowpar", ""), (124, 8, (128, 128), (256, 64), 64, "tiles", "observation wider than 123"),
    (24, 8, (256, 256), (256, 256), 64, "rowpar", ""), (24, 9, (256, 256), (256, 256), 64, "tiles", "action dimension above 8"),
    (24, 4, (96, 96), (96, 96), 64, "tiles", "hidden width not 64/128/256"),
    (24, 4, (256, 256), (256, 256), 512, "rowpar", ""), (24, 4, (256, 256), (256, 256), 513, "tiles", "batch above 512: the tile-parallel kernel is faster"),
    # eligible by shape, refused at set-up: the shared memory of the widest shapes, the program tables of 5 critic layers
    (100, 4, (256, 256), (256, 256), 64, "rowpar", ""), (101, 4, (256, 256), (256, 256), 64, "tiles", "shared memory budget exceeded"),
    (12, 2, (64,) * 4, (64,) * 4, 64, "rowpar", ""), (12, 2, (64,) * 2, (64,) * 5, 64, "tiles", "program tables too small"),
])
def test_rowpar_eligibility_boundaries(obs, act, hp, hq, B, kind, why, monkeypatch):
    """Which kernel a shape gets, at both sides of every limit, and the reason a refused shape reports. An update on a refused
    shape runs the tile-parallel kernel (tested elsewhere)."""
    from sac.engine import UpdateEngine
    monkeypatch.delenv("SACX_ROWPAR", raising=False)
    eng = UpdateEngine(obs, act, base_config(hidden=hp, q_hidden=hq, batch=B))
    assert eng.path() == (kind, why)
